"""
Oracle of the discovered-locus rule (tredparse_b200.strprofile.locus_for, DESIGN §4.5): from a region row of the
cohort outlier table and the reference sequence to the locus row the genotyper reads, restated in plain Python by
brute force over a dict {contig: sequence}.  It shares no code with the package.

  * candidate units: the k rotations of the row's motif m (period k) and the k rotations of its reverse complement;
  * tract: in the window [start - window, end + window) clipped to the contig, the longest run of exact, back-to-back
    copies of one candidate unit; ties go to the run whose centre is closest to the region's centre, then to the
    leftmost run; fewer than min_ref_units copies: no tract;
  * locus row: repeat = the unit at the tract's first base, repeat_location = contig:first-last (1-based, inclusive),
    18-base prefix / suffix (they must lie on the contig and hold only A, C, G, T), cut-offs ceil(read_length / k),
    name <contig>_<first>_<repeat>.
"""
import math

FLANK = 18
_RC = {"A": "T", "C": "G", "G": "C", "T": "A"}


def revcomp(s):
    return "".join(_RC[c] for c in reversed(s))


def tract(seq, lo, motif, start, end, min_ref_units=3):
    """(first base 0-based, unit, copies) of the tract of `motif` in seq, whose first base is at contig position lo;
    None without one"""
    k = len(motif)
    units = set()
    for m in (motif, revcomp(motif)):
        for i in range(k):
            units.add(m[i:] + m[:i])
    runs = []
    for u in units:
        for i in range(len(seq)):
            if i >= k and seq[i - k:i] == u:
                continue                                    # not the first copy of its run
            c = 0
            while seq[i + c * k:i + (c + 1) * k] == u:
                c += 1
            if c:
                runs.append((lo + i, u, c))
    if not runs:
        return None
    centre2 = start + end                                   # twice the region's centre
    best = min(runs, key=lambda r: (-r[2], abs(2 * r[0] + r[2] * k - centre2), r[0]))
    return best if best[2] >= min_ref_units else None


def locus(row, contigs, read_length, window=1000, min_ref_units=3):
    """-> (name, locus row with the hg38 location field) or the reason the row is skipped"""
    if row["contig"] == "-":
        return "no position"
    if row["contig"] not in contigs:
        return "contig not in FASTA"
    seq = contigs[row["contig"]].upper()
    motif = row["motif"]
    k = len(motif)
    lo, hi = max(0, row["start"] - window), min(len(seq), row["end"] + window)
    t = tract(seq[lo:hi], lo, motif, row["start"], row["end"], min_ref_units)
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
