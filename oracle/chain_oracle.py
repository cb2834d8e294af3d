"""
Plain-Python restatement of the interrupted-tract rule (tredsw_ref_tracts_ex, csrc/ref_tracts_device.cuh
`tract_chains`, DESIGN §4.5.1) and of the discovered-locus rule in chain mode (strprofile.locus_for with
max_interrupt >= 1), for the tests.  Nothing under tredparse_b200/ imports it, and it shares no code with the package:
it builds on the pure-rule oracles (tract_oracle.py, locus_oracle.py), which it leaves unchanged.

  * ag(j): s[j] and s[j + k] both in ACGT (any case) and equal; a run is a maximal [a, e) of ag = 1, a segment a run
    with e - a >= k;
  * segment S = [a, e) links to the next segment T = [a', e') when max_interrupt >= 1, both have root period k and
    one canonical code, a' - (e + k) <= max_interrupt and s[e + k:a'] holds only ACGT;
  * a chain S1 -> ... -> Sm gives [a1, a1 + c k), c = (em + k - a1) // k, with m segments, when A den >= num (em - a1)
    (A: ag = 1 in [a1, em)); a chain of m >= 2 failing that gives its segments alone;
  * kept: root period k, c >= min_units, c k >= min_len, requested code;
  * locus: the longest kept tract (in copies) of the row's motif in the window's text, min_len 0; ties as the pure
    rule's (centre, then leftmost); the rest of the row as locus_oracle.locus.
"""
import math

from .locus_oracle import FLANK
from .tract_oracle import canonical, code, root_period


def chained_tracts(contigs, motifs, min_units=3, min_len=30, max_interrupt=0, num=9, den=10):
    """contigs: {name: text of its bases} in FASTA order; motifs: strings.  -> [(contig index, start, length, period,
    canonical code, segments)] by (contig, start, period); with max_interrupt 0, tract_oracle.tracts with segments 1"""
    want = {(len(m), canonical(m.upper())) for m in motifs}
    out = []
    for ci, seq in enumerate(contigs.values()):
        s = seq.upper()
        n = len(s)
        for k in sorted({k for k, _ in want}):
            ag = [j + k < n and s[j] in "ACGT" and s[j] == s[j + k] for j in range(n)]
            segs, j = [], 0
            while j < n:
                if not ag[j]:
                    j += 1
                    continue
                a = j
                while j < n and ag[j]:
                    j += 1
                if j - a >= k:
                    unit = s[a:a + k]
                    segs.append((a, j, root_period(unit) == k and canonical(unit)))
            chains = []
            for a, e, cu in segs:
                last = chains[-1][-1] if chains else None
                if (max_interrupt > 0 and last is not None and cu and last[2] == cu
                        and a - (last[1] + k) <= max_interrupt
                        and all(b in "ACGT" for b in s[last[1] + k:a])):
                    chains[-1].append((a, e, cu))
                else:
                    chains.append([(a, e, cu)])
            for ch in chains:
                cu = ch[0][2]
                if not cu or (k, cu) not in want:
                    continue
                a1, em = ch[0][0], ch[-1][1]
                if sum(ag[a1:em]) * den >= num * (em - a1):
                    parts = [(a1, em, len(ch))]
                else:
                    parts = [(a, e, 1) for a, e, _ in ch]
                for a, e, m in parts:
                    c = (e + k - a) // k
                    if c >= min_units and c * k >= min_len:
                        out.append((ci, a, c * k, k, code(cu), m))
    return sorted(out, key=lambda t: (t[0], t[1], t[3]))


def tract(seq, lo, motif, start, end, min_ref_units=3, max_interrupt=1, purity=(9, 10)):
    """(first base 0-based, unit, copies) of the longest kept chain tract of `motif` in seq, whose first base is at
    contig position lo; None without one"""
    k = len(motif)
    found = chained_tracts({"w": seq}, [motif], min_ref_units, 0, max_interrupt, *purity)
    runs = [(lo + s, seq[s:s + k], n // k) for _, s, n, _, _, _ in found]
    if not runs:
        return None
    return min(runs, key=lambda r: (-r[2], abs(2 * r[0] + r[2] * k - start - end), r[0]))


def locus(row, contigs, read_length, window=1000, min_ref_units=3, max_interrupt=1, purity=(9, 10)):
    """-> (name, locus row with the hg38 location field) or the reason the row is skipped"""
    if row["contig"] == "-":
        return "no position"
    if row["contig"] not in contigs:
        return "contig not in FASTA"
    seq = contigs[row["contig"]].upper()
    motif = row["motif"]
    k = len(motif)
    lo, hi = max(0, row["start"] - window), min(len(seq), row["end"] + window)
    t = tract(seq[lo:hi], lo, motif, row["start"], row["end"], min_ref_units, max_interrupt, purity)
    if t is None:
        return "no reference tract"
    first, unit, copies = t
    last = first + copies * k                               # exclusive
    if first - FLANK < 0 or last + FLANK > len(seq):
        return "flank outside contig"
    prefix, suffix = seq[first - FLANK:first], seq[last:last + FLANK]
    if any(c not in "ACGT" for c in prefix + suffix):
        return "N in flank"
    name = "{}_{}_{}".format(row["contig"], first + 1, unit)
    cut = int(math.ceil(read_length / float(k)))
    return name, {"repeat": unit, "repeat_location": "{}:{}-{}".format(row["contig"], first + 1, last),
                  "prefix": prefix, "suffix": suffix, "inheritance": "AD", "mutation_nature": "increase",
                  "cutoff_prerisk": cut, "cutoff_risk": cut}
