"""
Synthetic (sample, locus) problems: reads simulated at a TRED locus for a given allele pair, plus the
paired-end distances the caller uses — the inputs of the hot path without a BAM in between.

Design follows SURVEY.md §8(d) (configs 3-5 of BASELINE.json):

* haplotype = rand(FLANK) + prefix18 + motif x h + suffix18 + rand(FLANK)   (random flanks: no hg38 here)
* 150 bp (or 250 bp) paired-end reads, fragment length N(350, 75^2) truncated to [200, 999], 15x per
  haplotype, 0.5 %/base substitution error, read 2 reverse-complemented;
* the read set of a problem = reads whose leftmost base lies within READLEN of the repeat (the rule of
  tredparse/bam_parser.py:206-214 in haplotype coordinates) — reads lying wholly inside a long repeat
  are included, they are the "unmapped with anchored mate" class;
* target_lens = fragment - (h - ref_copy) * period for pairs whose read 1 starts > 9 bp before and whose
  read 2 ends > 9 bp after the repeat (bam_parser.py:341-359), kept if < 1000;
  global_lens = 2,500 draws of the fragment distribution.

Everything is seeded: ``np.random.default_rng(0xB200 + 1000 * locus_idx + pair_idx)`` per problem.
"""
import numpy as np

from .ssw import encode

FLANK_BP = 2000
FRAG_MEAN, FRAG_SD, FRAG_MIN, FRAG_MAX = 350.0, 75.0, 200, 999
N_GLOBAL = 2500
_COMP = np.array([3, 2, 1, 0, 4], dtype=np.int8)


class Problem:
    """One (sample, locus) problem ready for the GPU path."""
    __slots__ = ("tred", "readlen", "ploidy", "depth", "reads", "roff", "global_lens", "target_lens",
                 "alleles", "names")

    def name_strings(self):
        return ["f{}".format(int(x)) for x in self.names]

    @property
    def nreads(self):
        return len(self.roff) - 1

    def read_strings(self):
        lut = np.array(list("ACGTN"))
        return ["".join(lut[self.reads[self.roff[i]:self.roff[i + 1]]]) for i in range(self.nreads)]


def _fragment_lengths(rng, n):
    out = np.empty(0, dtype=np.int64)
    while len(out) < n:
        x = np.rint(rng.normal(FRAG_MEAN, FRAG_SD, size=int((n - len(out)) * 1.3) + 8)).astype(np.int64)
        out = np.concatenate([out, x[(x >= FRAG_MIN) & (x <= FRAG_MAX)]])
    return out[:n]


def simulate_problem(tred, alleles, readlen=150, cov_per_hap=15.0, error=0.005, seed=0, depth=None):
    """alleles: (h1, h2) in repeat units for a diploid problem, (h,) for a haploid one."""
    rng = np.random.default_rng(seed)
    prefix, suffix, motif = encode(tred.prefix), encode(tred.suffix), encode(tred.repeat)
    P = len(motif)
    ref_copy = tred.ref_copy
    reads, target, names = [], [], []
    for hap_idx, h in enumerate(alleles):
        rep = np.tile(motif, h)
        nmask = rep == 4                               # 'N' in the motif (GCN loci): any base
        if nmask.any():
            rep = rep.copy()
            rep[nmask] = rng.integers(0, 4, int(nmask.sum()))
        hap = np.concatenate([rng.integers(0, 4, FLANK_BP).astype(np.int8), prefix, rep.astype(np.int8), suffix,
                              rng.integers(0, 4, FLANK_BP).astype(np.int8)])
        rep_start = FLANK_BP + len(prefix)
        rep_end = rep_start + P * h                   # exclusive
        L = len(hap)
        nfrag = int(round(cov_per_hap * L / (2.0 * readlen)))
        frag = _fragment_lengths(rng, nfrag)
        start = rng.integers(0, L - frag + 1)
        end = start + frag                             # exclusive
        # read 1: forward from the fragment start; read 2: reverse complement of the fragment end
        s1 = start
        s2 = end - readlen
        lo, hi = rep_start - readlen, rep_end + readlen
        k1 = (s1 >= lo) & (s1 <= hi)
        k2 = (s2 >= lo) & (s2 <= hi)
        idx = np.arange(readlen)
        r1 = hap[s1[k1][:, None] + idx]
        r2 = _COMP[hap[s2[k2][:, None] + idx]][:, ::-1]
        for block, kept in ((r1, k1), (r2, k2)):
            if block.size:
                # mates share a name: <haplotype>.<fragment> (remove_pairs_of_rept pairs reads by name)
                names.append(hap_idx * 1000000 + np.nonzero(kept)[0])
                err = rng.random(block.shape) < error
                block = np.where(err, rng.integers(0, 4, block.shape), block).astype(np.int8)
                reads.append(block)
        span = (s1 < rep_start - 9) & (end > rep_end + 9)
        tl = frag[span] - (h - ref_copy) * P
        target.append(tl[tl < 1000])
    pr = Problem()
    pr.tred, pr.readlen, pr.ploidy, pr.alleles = tred, readlen, len(alleles), tuple(alleles)
    allr = np.concatenate(reads) if reads else np.zeros((0, readlen), dtype=np.int8)
    order = rng.permutation(len(allr))                # BAM order mixes haplotypes and mates
    allr = allr[order]
    pr.reads = np.ascontiguousarray(allr.reshape(-1))
    pr.roff = np.arange(len(allr) + 1, dtype=np.int64) * readlen
    pr.global_lens = _fragment_lengths(rng, N_GLOBAL).astype(np.int32)
    pr.target_lens = (np.concatenate(target) if target else np.zeros(0)).astype(np.int32)
    pr.depth = float(depth) if depth is not None else cov_per_hap * len(alleles)
    pr.names = (np.concatenate(names)[order] if names else np.zeros(0, dtype=np.int64)).astype(np.int64)
    return pr


def draw_allele(rng, tred, risk_fraction=0.01):
    """One allele (units) from the locus' population histogram (TREDs.meta.csv allele_freq), with a
    small fraction forced into the risk range (SURVEY.md §8d config 4)."""
    freq = tred.allele_freq
    if rng.random() < risk_fraction or not freq:
        base = int(tred.cutoff_risk)
        return max(1, base + int(rng.integers(0, 30))) if tred.is_expansion else max(1, base - int(rng.integers(0, 3)))
    keys = np.array(sorted(freq))
    p = np.array([freq[k] for k in keys], dtype=float)
    return int(rng.choice(keys, p=p / p.sum()))


def cohort_specs(repo, names, nsamples, readlen=150, seed=20240000, maxunits=None, first_sample=0):
    """Specs (keyword arguments of ``simulate_from_spec``) of nsamples x len(names) problems: alleles drawn per
    sample from each locus' allele_freq; gender 50/50 (X-linked loci are haploid in males); depth ~ N(35, 5^2).
    Sample ``s`` depends on ``seed + s`` only, so ranks can simulate disjoint sample ranges independently."""
    specs = []
    for s in range(first_sample, first_sample + nsamples):
        rng = np.random.default_rng(seed + s)
        male = rng.random() < 0.5
        depth = float(np.clip(rng.normal(35, 5), 15, 60))
        for li, name in enumerate(names):
            tred = repo[name]
            ploidy = 1 if (male and tred.is_xlinked) else 2
            alleles = tuple(sorted(draw_allele(rng, tred) for _ in range(ploidy)))
            if maxunits:
                alleles = tuple(min(a, maxunits) for a in alleles)
            specs.append({"tred": name, "alleles": [int(a) for a in alleles], "readlen": readlen,
                          "cov_per_hap": depth / 2.0, "seed": 0xB200 + 1000 * li + 7919 * s, "sample": s})
    return specs


def sample_header(seed, s):
    """(male, depth) of cohort sample `s`: gender 50/50, depth ~ N(35, 5^2) clipped to [15, 60]."""
    rng = np.random.default_rng(seed + s)
    male = bool(rng.random() < 0.5)
    return male, float(np.clip(rng.normal(35, 5), 15, 60))


def problem_spec(repo, names, s, li, readlen=150, seed=20240000, maxunits=None):
    """Spec of the (sample s, locus li) problem of the cohort, independent of every other problem (own random
    stream), so that a rank can materialise exactly the problems it owns — same distribution as cohort_specs."""
    male, depth = sample_header(seed, s)
    tred = repo[names[li]]
    ploidy = 1 if (male and tred.is_xlinked) else 2
    rng = np.random.default_rng([seed + s, li, 0xA11E1E])
    alleles = tuple(sorted(draw_allele(rng, tred) for _ in range(ploidy)))
    if maxunits:
        alleles = tuple(min(a, maxunits) for a in alleles)
    return {"tred": names[li], "alleles": [int(a) for a in alleles], "readlen": readlen, "cov_per_hap": depth / 2.0,
            "seed": 0xB200 + 1000 * li + 7919 * s, "sample": s, "locus": li}


def problem_costs(repo, names, nsamples, readlen=150, seed=20240000, first_sample=0):
    """A-priori cost of every (sample, locus) problem, float64 [nsamples, nloci]: expected reads (depth x ploidy)
    x forward cells of the locus' template family — what a scheduler knows before reading a BAM (SURVEY §8e)."""
    cells = np.zeros(len(names))
    xl = np.zeros(len(names), dtype=bool)
    for li, n in enumerate(names):
        t = repo[n]
        P, flank = len(t.repeat), len(t.prefix) + len(t.suffix)
        mu = -(-readlen // P)
        cells[li] = 2.0 * readlen * sum(flank + P * u for u in range(1, mu + 1))
        xl[li] = t.is_xlinked
    out = np.zeros((nsamples, len(names)))
    for k in range(nsamples):
        male, depth = sample_header(seed, first_sample + k)
        out[k] = depth * np.where(xl & male, 0.5, 1.0) * cells
    return out


def simulate_from_spec(repo, spec):
    return simulate_problem(repo[spec["tred"]], tuple(spec["alleles"]), readlen=spec.get("readlen", 150),
                            cov_per_hap=spec.get("cov_per_hap", 15.0), error=spec.get("error", 0.005),
                            seed=spec["seed"], depth=spec.get("depth"))


def simulate_cohort(repo, names, nsamples, readlen=150, seed=20240000, maxunits=None, first_sample=0):
    return [simulate_from_spec(repo, sp) for sp in
            cohort_specs(repo, names, nsamples, readlen, seed, maxunits, first_sample)]


# ---------------------------------------------------------------------------------------------------------
# the same simulation as aligned records: synthetic whole-sample BAMs for the from-BAM path
# ---------------------------------------------------------------------------------------------------------
def locus_records(tred, tid, alleles, readlen=150, cov_per_hap=15.0, error=0.005, seed=0, tag="", flank=FLANK_BP):
    """Paired reads of one locus as ``bamio.AlignedSegment`` records placed on the reference: haplotype coordinates are
    mapped onto the locus (flanks one to one, the repeat clamped to the reference's copy number), every read gets a
    ``<readlen>M`` CIGAR and proper-pair flags — what an aligner reports for reads around a repeat whose length
    differs from the reference.  Haplotypes, fragment lengths and errors follow the model of ``simulate_problem``
    (not its random stream).  A fragment shorter than the read is dropped: an aligner would not report it as a
    full-length ``<readlen>M`` proper pair.  Fragments are at least FRAG_MIN long, so for ``readlen <= FRAG_MIN``
    nothing is dropped and the records do not depend on this rule."""
    from .bamio import AlignedSegment
    rng = np.random.default_rng(seed)
    prefix, suffix, motif = encode(tred.prefix), encode(tred.suffix), encode(tred.repeat)
    P = len(motif)
    lut = np.array(list("ACGTN"))
    recs = []
    ref_rep_len = tred.repeat_end - tred.repeat_start + 1
    for hap_idx, h in enumerate(alleles):
        rep = np.tile(motif, h)
        nmask = rep == 4
        if nmask.any():
            rep = rep.copy()
            rep[nmask] = rng.integers(0, 4, int(nmask.sum()))
        hap = np.concatenate([rng.integers(0, 4, flank).astype(np.int8), prefix, rep.astype(np.int8), suffix,
                              rng.integers(0, 4, flank).astype(np.int8)])
        rep_start = flank + len(prefix)
        rep_end = rep_start + P * h
        L = len(hap)
        nfrag = int(round(cov_per_hap * L / (2.0 * readlen)))
        frag = _fragment_lengths(rng, nfrag)
        start = rng.integers(0, L - frag + 1)
        end = start + frag
        full = np.nonzero(frag >= readlen)[0]             # then 0 <= start <= end - readlen and end <= L
        start, end = start[full], end[full]

        def to_ref(x):        # haplotype coordinate -> 0-based reference coordinate
            x = np.asarray(x)
            left = (tred.repeat_start - 1) - (rep_start - x)
            inside = (tred.repeat_start - 1) + np.minimum(x - rep_start, ref_rep_len - 1)
            right = tred.repeat_end + (x - rep_end)
            return np.where(x < rep_start, left, np.where(x < rep_end, inside, right))
        s1, s2 = start, end - readlen
        p1, p2 = to_ref(s1), to_ref(s2)
        e2 = to_ref(end - 1) + 1
        idx = np.arange(readlen)
        r1 = hap[s1[:, None] + idx]
        r2 = hap[s2[:, None] + idx]                     # stored on the forward strand, flagged reverse
        for block in (r1, r2):
            err = rng.random(block.shape) < error
            block[err] = rng.integers(0, 4, int(err.sum()))
        for k, fk in enumerate(full):
            name = "{}h{}f{}".format(tag, hap_idx, fk)
            tl = int(e2[k] - p1[k])
            recs.append(AlignedSegment(name, 0x1 | 0x2 | 0x20 | 0x40, tid, int(p1[k]), 60, [(0, readlen)], tid, int(p2[k]),
                                       tl, "".join(lut[r1[k]])))
            recs.append(AlignedSegment(name, 0x1 | 0x2 | 0x10 | 0x80, tid, int(p2[k]), 60, [(0, readlen)], tid, int(p1[k]),
                                       -tl, "".join(lut[r2[k]])))
    return recs


def write_sample_bam(path, repo, names, references, sample, readlen=150, seed=20240000, flank=10000):
    """One synthetic sample as an indexed BAM: paired reads in a +-`flank` window (default 10 kb: the reference's
    paired-end window, bam_parser.py:31) around every locus of `names`,
    alleles / gender / depth as in ``problem_spec``.  references: [(contig, length)] of the header.
    :return: {tred name: alleles} (the truth)"""
    from .bamio import write_bam
    tid = {n: i for i, (n, _) in enumerate(references)}
    recs, truth = [], {}
    for li, name in enumerate(names):
        sp = problem_spec(repo, names, sample, li, readlen, seed)
        t = repo[name]
        if t.chr not in tid:
            continue
        truth[name] = sp["alleles"]
        recs += locus_records(t, tid[t.chr], tuple(sp["alleles"]), readlen, sp["cov_per_hap"], seed=sp["seed"],
                              tag="s{}l{}".format(sample, li), flank=flank)
    recs.sort(key=lambda r: (r.reference_id, r.reference_start))
    write_bam(path, references, recs, level=1)
    return truth


# ---------------------------------------------------------------------------------------------------------
# planted expansions anywhere: the in-repeat reads of the STR profile (strprofile)
# ---------------------------------------------------------------------------------------------------------
def _mq_aux(mq):
    """the raw aux bytes of an MQ:i tag (stored as type C, as aligners write small values)"""
    return b"MQC" + bytes([mq])


def expansion_records(tid, pos, motif, units, readlen=150, cov=15.0, flank=2000, error=0.005, seed=0, tag="x",
                      mq_tags=True, mismap_fraction=0.0, mismap_to=None):
    """Paired reads of a haplotype with `units` copies of `motif` inserted at 0-based reference position `pos` of contig
    `tid` (random flanks of `flank` bases on either side, mapped one to one onto [pos - flank, pos + flank)), placed as
    an aligner places reads around an expansion longer than a read:
      * pairs with no read inside the repeat: proper pairs, MAPQ 60, ``<readlen>M``;
      * a read wholly inside the repeat (an in-repeat read) whose mate is not: unmapped, placed at its mate's position
        (tid / pos / next = the mate's), its mate flagged 0x8; with probability `mismap_fraction` it is instead mismapped
        at MAPQ 0 at a random position of ``mismap_to = (tid, start, end)``, its mate pointing there;
      * both reads inside the repeat: both unmapped, in the unmapped tail (tid -1).
    The in-repeat read carries its mate's MAPQ as an ``MQ`` tag (mapped mates carry one too) unless ``mq_tags`` is
    False.  Records are bamio.AlignedSegment, not sorted (``coordinate_sort``); write them with
    ``bamio.write_bam(..., aux=True)`` to keep the MQ tags."""
    from .bamio import AlignedSegment
    rng = np.random.default_rng(seed)
    m = encode(motif)
    rep = np.tile(m, units).astype(np.int8)
    hap = np.concatenate([rng.integers(0, 4, flank).astype(np.int8), rep, rng.integers(0, 4, flank).astype(np.int8)])
    rep_start, rep_end, L = flank, flank + len(rep), len(hap)
    lut = np.array(list("ACGTN"))
    nfrag = int(round(cov * L / (2.0 * readlen)))
    frag = _fragment_lengths(rng, nfrag)
    frag = frag[frag >= readlen]
    start = rng.integers(0, L - frag + 1)

    def to_ref(x):
        return pos - (rep_start - x) if x < rep_start else (pos if x < rep_end else pos + (x - rep_end))
    aux = (lambda q: _mq_aux(q)) if mq_tags else (lambda q: b"")
    recs = []
    for k in range(len(frag)):
        s1, s2 = int(start[k]), int(start[k] + frag[k] - readlen)
        seqs = []
        for s_ in (s1, s2):
            r = hap[s_:s_ + readlen].copy()
            err = rng.random(readlen) < error
            r[err] = rng.integers(0, 4, int(err.sum()))
            seqs.append("".join(lut[r]))
        irr = [s_ >= rep_start and s_ + readlen <= rep_end for s_ in (s1, s2)]
        p = [to_ref(s1), to_ref(s2)]
        seg, strand = (0x40, 0x80), (0x20, 0x10)
        name = "{}f{}".format(tag, k)
        if not irr[0] and not irr[1]:
            for i in (0, 1):
                recs.append(AlignedSegment(name, 0x1 | 0x2 | seg[i] | strand[i], tid, p[i], 60, [(0, readlen)], tid,
                                           p[1 - i], 0, seqs[i], aux=aux(60)))
        elif irr[0] and irr[1]:
            for i in (0, 1):
                recs.append(AlignedSegment(name, 0x1 | 0x4 | 0x8 | seg[i] | strand[i], -1, -1, 0, [], -1, -1, 0, seqs[i]))
        else:
            i, j = (0, 1) if irr[0] else (1, 0)              # i: the in-repeat read, j: its anchor
            if mismap_to is not None and rng.random() < mismap_fraction:
                mt, ms, me = mismap_to
                mp = int(rng.integers(ms, me))
                recs.append(AlignedSegment(name, 0x1 | seg[i] | strand[i], mt, mp, 0, [(0, readlen)], tid, p[j], 0,
                                           seqs[i], aux=aux(60)))
                recs.append(AlignedSegment(name, 0x1 | seg[j] | strand[j], tid, p[j], 60, [(0, readlen)], mt, mp, 0,
                                           seqs[j], aux=aux(0)))
            else:
                recs.append(AlignedSegment(name, 0x1 | 0x4 | seg[i] | strand[i], tid, p[j], 0, [], tid, p[j], 0,
                                           seqs[i], aux=aux(60)))
                recs.append(AlignedSegment(name, 0x1 | 0x8 | seg[j] | strand[j], tid, p[j], 60, [(0, readlen)], tid,
                                           p[j], 0, seqs[j]))
    return recs


def coordinate_sort(recs):
    """records in coordinate order: by contig, then position; unmapped records without a contig (tid -1) last"""
    return sorted(recs, key=lambda r: (r.reference_id if r.reference_id >= 0 else 1 << 31, r.reference_start))


# ---------------------------------------------------------------------------------------------------------
# a reference and reads that agree with it: discovered loci (strprofile.locus_for) end to end
# ---------------------------------------------------------------------------------------------------------
def planted_reference(lengths, sites, seed=0):
    """Random contigs {name: bases} of `lengths` [(name, length)] with repeat tracts planted: a site (contig, pos,
    unit, copies) writes `copies` back-to-back copies of `unit` from 0-based `pos` on.  The base before a tract is
    not the unit's last base and the base after it not its first, so no rotation of the unit runs longer: the tract is
    exactly the planted one."""
    rng = np.random.default_rng(seed)
    seqs = {n: rng.choice(list("ACGT"), L) for n, L in lengths}
    for contig, pos, unit, copies in sites:
        s, end = seqs[contig], pos + len(unit) * copies
        s[pos:end] = list(unit * copies)
        if pos > 0 and s[pos - 1] == unit[-1]:
            s[pos - 1] = "ACGT"[("ACGT".index(unit[-1]) + 1) % 4]
        if end < len(s) and s[end] == unit[0]:
            s[end] = "ACGT"[("ACGT".index(unit[0]) + 1) % 4]
    return {n: "".join(s) for n, s in seqs.items()}


def write_fasta(path, contigs, width=60, fai=False):
    """contigs {name: bases} as a FASTA of `width` bases a line; with `fai`, its samtools-style index at path.fai"""
    rows, offset = [], 0
    with open(path, "w") as fp:
        for name, seq in contigs.items():
            head = ">{}\n".format(name)
            fp.write(head)
            lb = min(width, len(seq))                        # (a record of one short line: its own width)
            rows.append("{}\t{}\t{}\t{}\t{}\n".format(name, len(seq), offset + len(head), lb, lb + 1 if lb else 0))
            body = "".join(seq[i:i + width] + "\n" for i in range(0, len(seq), width))
            fp.write(body)
            offset += len(head) + len(body)
    if fai:
        with open(path + ".fai", "w") as fp:
            fp.writelines(rows)
    return path


def reference_records(seq, tid, rep_start, rep_end, motif, alleles, readlen=150, cov_per_hap=15.0, flank=2000,
                      error=0.005, seed=0, tag=""):
    """Paired reads of a locus whose reference tract is seq[rep_start:rep_end] (0-based): haplotype h = the reference's
    `flank` bases before the tract, h copies of `motif`, its `flank` bases after the tract.  Fragment lengths and
    errors follow ``locus_records``; reads are placed as ``locus_records`` and ``expansion_records`` place them:
      * pairs with no read wholly inside the repeat: ``<readlen>M`` proper pairs, MAPQ 60, flanks mapped one to one
        and the repeat clamped to the reference's tract;
      * an in-repeat read whose mate is not one: unmapped at its mate's position, the mate flagged 0x8;
      * both reads inside the repeat: both unmapped, in the unmapped tail (tid -1).
    Records with a mapped mate carry its MAPQ as an ``MQ`` tag.  Not sorted (``coordinate_sort``); write them with
    ``bamio.write_bam(..., aux=True)``."""
    from .bamio import AlignedSegment
    rng = np.random.default_rng(seed)
    lut = np.array(list("ACGTN"))
    ref_len = rep_end - rep_start
    left = encode(seq[max(0, rep_start - flank):rep_start])
    right = encode(seq[rep_end:rep_end + flank])
    recs = []
    for hap_idx, h in enumerate(alleles):
        hap = np.concatenate([left, np.tile(encode(motif), h), right]).astype(np.int8)
        hrs, hre, L = len(left), len(left) + len(motif) * h, len(left) + len(motif) * h + len(right)

        def to_ref(x):
            if x < hrs:
                return rep_start - (hrs - x)
            return rep_start + min(x - hrs, ref_len - 1) if x < hre else rep_end + (x - hre)
        nfrag = int(round(cov_per_hap * L / (2.0 * readlen)))
        frag = _fragment_lengths(rng, nfrag)
        frag = frag[(frag >= readlen) & (frag <= L)]
        start = rng.integers(0, L - frag + 1)
        for k in range(len(frag)):
            s = (int(start[k]), int(start[k] + frag[k] - readlen))
            seqs = []
            for s_ in s:
                r = hap[s_:s_ + readlen].copy()
                err = rng.random(readlen) < error
                r[err] = rng.integers(0, 4, int(err.sum()))
                seqs.append("".join(lut[r]))
            irr = [hrs <= s_ and s_ + readlen <= hre for s_ in s]
            p = [to_ref(s_) for s_ in s]
            seg, strand = (0x40, 0x80), (0x20, 0x10)
            name = "{}h{}f{}".format(tag, hap_idx, k)
            if not irr[0] and not irr[1]:
                tl = to_ref(s[1] + readlen - 1) + 1 - p[0]
                for i in (0, 1):
                    recs.append(AlignedSegment(name, 0x1 | 0x2 | seg[i] | strand[i], tid, p[i], 60, [(0, readlen)],
                                               tid, p[1 - i], tl if i == 0 else -tl, seqs[i], aux=_mq_aux(60)))
            elif irr[0] and irr[1]:
                for i in (0, 1):
                    recs.append(AlignedSegment(name, 0x1 | 0x4 | 0x8 | seg[i] | strand[i], -1, -1, 0, [], -1, -1, 0,
                                               seqs[i]))
            else:
                i, j = (0, 1) if irr[0] else (1, 0)          # i: the in-repeat read, j: its anchor
                recs.append(AlignedSegment(name, 0x1 | 0x4 | seg[i] | strand[i], tid, p[j], 0, [], tid, p[j], 0,
                                           seqs[i], aux=_mq_aux(60)))
                recs.append(AlignedSegment(name, 0x1 | 0x8 | seg[j] | strand[j], tid, p[j], 60, [(0, readlen)], tid,
                                           p[j], 0, seqs[j]))
    return recs
