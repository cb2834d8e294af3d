"""
STR profile of a whole BAM: the in-repeat reads (IRRs, reads made almost entirely of one short motif) of every record,
found on the GPU in one streaming scan of the file (``ingest.scan_sample(..., irr=IrrParams())``, DESIGN §4.5),
anchored by their mapped mates and merged into regions per motif; then a cohort comparison that ranks the samples
with more anchored IRRs in a region than the rest of the cohort — expansions outside the catalogue.

    prof = strprofile.profile("x.bam")                 # or "-" / a FIFO: read once, in order
    rows = strprofile.outliers([prof_a, prof_b, ...])  # highest z first

    python -m tredparse_b200.strprofile profile x.bam [y.bam ... | -] --workdir w
    python -m tredparse_b200.tred samples.csv --workdir w --str-profile     # or: catalogue calls and profiles, one read
    python -m tredparse_b200.strprofile outliers w/*.str_profile.json --tsv out.tsv
    python -m tredparse_b200.strprofile loci out.tsv --fasta ref.fa[.gz] --profiles w/*.str_profile.json [--alts]
        [--max-interruption N]
    python -m tredparse_b200.tred samples.csv --tred <name> ...          # from the directory that holds sites/

Definitions (include/tredsw.h, tredsw_irr_params):
  * an IRR record is primary (0x100, 0x200, 0x400, 0x800 unset), mapped or not, at least ``min_read_len`` long, and
    periodic at some period in [min_period, max_period] with purity num / den; its canonical motif is the smallest
    rotation of its motif and of the motif's reverse complement;
  * a paired IRR is a pair (one name, segment flags 0x40 / 0x80) of IRRs of the same motif;
  * an anchored IRR is paired (0x1), its mate is mapped (0x8 unset) and not an IRR, and its MQ tag, when it has one, is
    at least ``min_anchor_mapq``: its anchor is its (next_refID, next_pos).  Without an MQ tag it is counted (and so
    is ``anchors_without_mq``): the mate's MAPQ is not on the record and the scan reads every record once;
  * depth = bases of the primary, mapped, non-duplicate, non-QC-fail records / the summed contig lengths of the
    reference dictionary (the @SQ LN values); a normalised count is count x 40 / depth.
"""
import argparse
import json
import math
import os
import sys

from . import _lib
from .fasta import MIN_REF_UNITS, MIN_TRACT_LEN
from .ingest import BamIngest, IrrParams, is_stream, scan_sample

MIN_ANCHOR_MAPQ = 50
MERGE_DISTANCE = 500
NORM_DEPTH = 40.0
LOCUS_WINDOW = 1000
LOCUS_FLANK = 18
ALT_SPAN = 1000         # a locus' own read window: its tract +- this many bases
MAX_ALTS = 100          # the catalogue's largest count of alt regions (FXTAS)
_RC = str.maketrans("ACGT", "TGCA")


def motif_string(period, bits):
    """the bases of a motif of `period` bases, 2 bits each, first base most significant"""
    return "".join("ACGT"[(bits >> (2 * (period - 1 - i))) & 3] for i in range(period))


def sample_key(path, handle):
    """the sample key tred.py uses: the @RG SM of stdin ("stdin" without one), else the file name without extension"""
    if path == "-":
        return handle.read_group_sample() or "stdin"
    return os.path.basename(path).rsplit(".", 1)[0]


def build_profile(irr, refs, params, min_anchor_mapq=MIN_ANCHOR_MAPQ, merge_distance=MERGE_DISTANCE, sample=None,
                  bam=None):
    """the profile dict from the IRR entries of a scan (``ScanBatch.irr``)"""
    ent, st0 = irr["entries"], irr["stats"]
    st = dict(st0, anchors_below_mapq=0, anchored_irrs=0, paired_irrs=0, irr_pairs_motif_mismatch=0)
    counts, anchors = {}, {}
    for k, e in enumerate(ent.tolist()):
        tid, pos, next_tid, next_pos, flag, mapq, mq, period, motif, _, _, mate = e
        key = motif_string(period, motif)
        if mate >= 0:                                   # both reads are IRRs: a paired IRR (counted once, at read 1)
            if flag & 0x40:
                if (int(ent["period"][mate]), int(ent["motif"][mate])) == (period, motif):
                    counts.setdefault(key, [0, 0])[1] += 1
                    st["paired_irrs"] += 1
                else:
                    st["irr_pairs_motif_mismatch"] += 1
            continue
        if not (flag & 1) or (flag & 8) or next_tid < 0:
            continue
        if 0 <= mq < min_anchor_mapq:
            st["anchors_below_mapq"] += 1
            continue
        counts.setdefault(key, [0, 0])[0] += 1
        st["anchored_irrs"] += 1
        anchors.setdefault(key, []).append((next_tid, next_pos))
    prof = {}
    for key in sorted(counts):
        regions = []
        for tid, pos in sorted(anchors.get(key, ())):
            last = regions[-1] if regions else None
            if last is not None and last[0] == tid and pos - (last[2] - 1) <= merge_distance:
                last[2], last[3] = pos + 1, last[3] + 1
            else:
                regions.append([tid, pos, pos + 1, 1])
        prof[key] = {"anchored_irr_count": counts[key][0], "paired_irr_count": counts[key][1],
                     "regions": [{"contig": refs[t][0], "start": s, "end": e, "count": c} for t, s, e, c in regions]}
    total = sum(n for _, n in refs)
    return {"sample": sample, "bam": bam, "read_length": st["max_l_seq"],
            "depth": st["depth_bases"] / total if total else 0.0,
            "params": dict(params.as_dict(), min_anchor_mapq=min_anchor_mapq, merge_distance=merge_distance),
            "stats": st, "profile": prof}


def profile(path, ctx=None, sample=None, min_period=2, max_period=20, purity_num=9, purity_den=10, min_read_len=50,
            min_anchor_mapq=MIN_ANCHOR_MAPQ, merge_distance=MERGE_DISTANCE, slab_bytes=None, emulate=False):
    """The STR profile of one BAM from ONE scan on the GPU (``ctx``: a ``_lib.Context``, default the process's).
    ``-``, FIFOs and sockets are read once, in order (``BamIngest.stream``); anything else through
    ``BamIngest.unindexed`` (an index, if any, is not needed).  ``emulate`` runs the serial host emulation of the
    device code instead — test infrastructure only.  Raises IOError when the scan fails (I/O, BGZF framing, a block
    that does not inflate, corrupt records, a file not sorted by coordinate)."""
    params = IrrParams(min_period, max_period, purity_num, purity_den, min_read_len)
    h = BamIngest.stream(path) if is_stream(path) else BamIngest.unindexed(path)
    try:
        refs = h.references()
        if sample is None:
            sample = sample_key(path, h)
        with scan_sample(None if emulate else (ctx or _lib.default_context()), h, [], [], [], slab_bytes=slab_bytes,
                         irr=params) as b:
            if b.scan_status:
                raise IOError("the GPU scan of `{}` failed (status {}): {}".format(path, b.scan_status, _lib.last_error()))
            irr = b.irr
    finally:
        h.close()
    return build_profile(irr, refs, params, min_anchor_mapq, merge_distance, sample=sample, bam=path)


def write_profile(prof, path):
    """a profile as a <sample>.str_profile.json file (what ``outliers`` and ``loci --profiles`` read)"""
    with open(path, "w") as fp:
        json.dump(prof, fp, indent=1, sort_keys=True)
        fp.write("\n")


def _zscore(xs, i):
    """(x_i - mean of the others) / max(population sd of the others, 1)"""
    others = xs[:i] + xs[i + 1:]
    mean = sum(others) / len(others)
    sd = math.sqrt(sum((o - mean) ** 2 for o in others) / len(others))
    return (xs[i] - mean) / max(sd, 1.0)


def _outlier_row(contig, start, end, motif, samples, xs):
    zs = [_zscore(xs, i) for i in range(len(xs))]
    top = max(range(len(zs)), key=lambda i: (zs[i], -i))
    return {"contig": contig, "start": start, "end": end, "motif": motif, "top_sample": samples[top], "z": zs[top],
            "counts": dict(zip(samples, xs))}


def outliers(profiles, merge_distance=None):
    """Rows of the cohort comparison, highest z first: per motif, one row per cohort region (the union of the samples'
    regions, merged within merge_distance — default: the first profile's) with every sample's normalised anchored
    IRR count there, and one row (contig "-", start / end None) of normalised paired IRR counts.  z of a sample = (its
    count - the mean of the others) / max(the population sd of the others, 1); a row names its top sample."""
    if len(profiles) < 2:
        raise ValueError("outliers: a cohort needs at least two samples (got {})".format(len(profiles)))
    samples = [p["sample"] for p in profiles]
    if len(set(samples)) != len(samples):
        raise ValueError("outliers: sample names repeat: {}".format(samples))
    md = profiles[0]["params"]["merge_distance"] if merge_distance is None else merge_distance
    scale = [NORM_DEPTH / p["depth"] if p["depth"] > 0 else 0.0 for p in profiles]
    rows = []
    for motif in sorted({m for p in profiles for m in p["profile"]}):
        regs = [p["profile"].get(motif, {}).get("regions", []) for p in profiles]
        merged = []
        for c, s, e in sorted((r["contig"], r["start"], r["end"]) for rs in regs for r in rs):
            if merged and merged[-1][0] == c and s - (merged[-1][2] - 1) <= md:
                merged[-1][2] = max(merged[-1][2], e)
            else:
                merged.append([c, s, e])
        for c, s, e in merged:
            xs = [sum(r["count"] for r in rs if r["contig"] == c and s <= r["start"] < e) * f for rs, f in zip(regs, scale)]
            rows.append(_outlier_row(c, s, e, motif, samples, xs))
        xs = [p["profile"].get(motif, {}).get("paired_irr_count", 0) * f for p, f in zip(profiles, scale)]
        rows.append(_outlier_row("-", None, None, motif, samples, xs))
    rows.sort(key=lambda r: (-r["z"], r["motif"], r["contig"], -1 if r["start"] is None else r["start"]))
    return rows


def write_tsv(rows, samples, fp):
    fp.write("\t".join(["contig", "start", "end", "motif", "top_sample", "z"] + list(samples)) + "\n")
    for r in rows:
        cells = [r["contig"], "-" if r["start"] is None else str(r["start"]), "-" if r["end"] is None else str(r["end"]),
                 r["motif"], r["top_sample"], "{:.4f}".format(r["z"])] + ["{:.4f}".format(r["counts"][s]) for s in samples]
        fp.write("\t".join(cells) + "\n")


def read_tsv(fp):
    """the rows of an ``outliers`` table (``write_tsv``): contig, start, end (None for a motif-only row), motif,
    top_sample, z and the per-sample counts"""
    header = fp.readline().rstrip("\n").split("\t")
    if header[:6] != ["contig", "start", "end", "motif", "top_sample", "z"]:
        raise ValueError("not an outliers table (header {})".format(header[:6]))
    rows = []
    for line in fp:
        c = line.rstrip("\n").split("\t")
        if len(c) < 6:
            continue
        rows.append({"contig": c[0], "start": None if c[1] == "-" else int(c[1]), "end": None if c[2] == "-" else int(c[2]),
                     "motif": c[3], "top_sample": c[4], "z": float(c[5]),
                     "counts": {s: float(x) for s, x in zip(header[6:], c[6:])}})
    return rows


class Skip(ValueError):
    """an outlier row that gives no locus; str() is the reason"""


def chain_tracts(seq, units, min_units, max_interrupt, purity):
    """The kept tracts of the interrupted-tract rule (DESIGN §4.5.1, as ``Fasta.tracts(..., max_interrupt)`` computes
    them on the GPU) in the text `seq` for one motif: `units` are the rotations of the motif and of its reverse
    complement, all of one period k with root period k.  -> [(start, copies)] in seq coordinates, at least
    `min_units` copies each."""
    k = len(next(iter(units)))
    num, den = purity
    n = len(seq)
    ag = [j + k < n and seq[j] in "ACGT" and seq[j] == seq[j + k] for j in range(n)]
    chains, j = [], 0                                   # chains of segments [(a, e)]; None: a segment of another code
    while j < n:
        if not ag[j]:
            j += 1
            continue
        a = j
        while j < n and ag[j]:
            j += 1
        if j - a < k:
            continue
        last = chains[-1] if chains else None
        if seq[a:a + k] not in units:
            chains.append(None)
        elif (last is not None and a - (last[-1][1] + k) <= max_interrupt
              and all(b in "ACGT" for b in seq[last[-1][1] + k:a])):
            last.append((a, j))
        else:
            chains.append([(a, j)])
    out = []
    for ch in chains:
        if ch is None:
            continue
        a1, em = ch[0][0], ch[-1][1]
        parts = [(a1, em)] if sum(ag[a1:em]) * den >= num * (em - a1) else ch
        out += [(a, (e + k - a) // k) for a, e in parts if (e + k - a) // k >= min_units]
    return out


def locus_for(row, fasta, read_length, window=LOCUS_WINDOW, min_ref_units=MIN_REF_UNITS, ref=None, max_interrupt=0,
              purity=(9, 10)):
    """The locus behind a region row of ``outliers`` -> (name, locus row for ``meta.TRED``); raises Skip(reason).

    Candidate units are the k rotations of the row's canonical motif (period k) and the k rotations of its reverse
    complement.  The tract is the longest run of exact, back-to-back copies of one candidate unit in the reference
    window [start - window, end + window) clipped to the contig: the region spans the anchors, mates that lie up to a
    fragment from the tract.  Ties go to the run whose centre is closest to the region's centre, then to the leftmost
    run.  Reasons to skip: ``no position`` (a motif-only row), ``contig not in FASTA``, ``no reference tract`` (fewer
    than `min_ref_units` copies), ``flank outside contig``, ``N in flank`` (any base but A, C, G, T in the 18 bases
    either side).

    With ``max_interrupt`` >= 1 the tract is instead the longest tract (in copies) of the row's motif that the
    interrupted-tract rule keeps in the window's text (``chain_tracts``: pure runs joined across interruptions of up
    to max_interrupt bases at `purity` (num, den), DESIGN §4.5.1), with the same ties; a motif whose root period is
    shorter than k has none.  Its prefix and suffix then lie outside the whole interrupted tract.

    The row: ``repeat`` = the unit as it reads on the reference at the tract's first base; the location
    ``contig:first-last`` (1-based, inclusive, the contig named as in the BAM header) under the field of `ref`
    (``meta.location_field``, default hg38); 18-base ``prefix`` / ``suffix``; inheritance AD, mutation_nature
    increase; ``cutoff_prerisk`` = ``cutoff_risk`` = ceil(read_length / k).  A discovered locus has no clinical
    cut-off: with this one, label ``risk`` and PP state that an allele is longer than a read, which is what an excess
    of anchored in-repeat reads supports.  The name is ``<contig>_<first>_<repeat>``."""
    from .meta import REF, location_field
    contig, motif = row["contig"], row["motif"]
    if contig == "-" or row.get("start") is None:
        raise Skip("no position")
    if contig not in fasta:
        raise Skip("contig not in FASTA")
    k = len(motif)
    length = fasta.lengths()[contig]
    lo, hi = max(0, row["start"] - window), min(length, row["end"] + window)
    seq = fasta.fetch(contig, lo, hi)
    rc = motif.translate(_RC)[::-1]
    units = {m[i:] + m[:i] for m in (motif, rc) for i in range(k)}
    centre2 = row["start"] + row["end"] - 2 * lo         # twice the region's centre, in window coordinates
    if max_interrupt:
        primitive = all(motif != motif[d:] + motif[:d] for d in range(1, k))
        found = chain_tracts(seq, units, min_ref_units, max_interrupt, purity) if primitive else []
        best = min(((-c, abs(2 * i + c * k - centre2), i) for i, c in found), default=None)
    else:
        # copies[i]: back-to-back copies of the candidate unit seq[i:i+k] from i on (right to left: one pass)
        copies = [0] * (len(seq) + k)
        for i in range(len(seq) - k, -1, -1):
            u = seq[i:i + k]
            if u in units:
                copies[i] = 1 + (copies[i + k] if seq[i + k:i + 2 * k] == u else 0)
        best = None
        for i in range(len(seq) - k + 1):
            c = copies[i]
            if c and not (i >= k and seq[i - k:i] == seq[i:i + k]):          # the first copy of a run
                key = (-c, abs(2 * i + c * k - centre2), i)
                if best is None or key < best:
                    best = key
    if best is None or -best[0] < min_ref_units:
        raise Skip("no reference tract")
    first, n = lo + best[2], -best[0]
    last = first + n * k                                 # exclusive
    if first - LOCUS_FLANK < 0 or last + LOCUS_FLANK > length:
        raise Skip("flank outside contig")
    prefix, suffix = fasta.fetch(contig, first - LOCUS_FLANK, first), fasta.fetch(contig, last, last + LOCUS_FLANK)
    if any(b not in "ACGT" for b in prefix + suffix):
        raise Skip("N in flank")
    repeat = seq[first - lo:first - lo + k]
    name = "{}_{}_{}".format(contig, first + 1, repeat)
    cut = -(-int(read_length) // k)
    return name, {"title": "Discovered {} repeat".format(motif), "gene_name": "", "id": name, "motif": motif,
                  "repeat": repeat, location_field(ref or REF): "{}:{}-{}".format(contig, first + 1, last),
                  "prefix": prefix, "suffix": suffix, "inheritance": "AD", "mutation_nature": "increase",
                  "cutoff_prerisk": cut, "cutoff_risk": cut}


def discover_loci(rows, fasta, read_length, min_z=3.0, window=LOCUS_WINDOW, min_ref_units=MIN_REF_UNITS, ref=None,
                  max_interrupt=0, purity=(9, 10)):
    """The loci of the outlier rows with z >= min_z, in row order -> ({name: locus row}, [(row, reason)] of the rows
    skipped).  Rows that resolve to one (contig, first base, repeat) — the left and right anchors of a long expansion
    can make two regions — give one locus, the first row's.  ``max_interrupt`` and ``purity``: ``locus_for``."""
    sites, skipped = {}, []
    for row in rows:
        if row["z"] < min_z:
            continue
        try:
            name, locus = locus_for(row, fasta, read_length, window, min_ref_units, ref, max_interrupt, purity)
        except Skip as e:
            skipped.append((row, str(e)))
            continue
        sites.setdefault(name, locus)
    return sites, skipped


def alt_regions_for(locus_row, tracts, read_length, max_alts=MAX_ALTS, ref=None):
    """The alt regions of a locus row (``locus_for``), from the tracts of a reference scan (``Fasta.tracts``): the
    regions an aligner may place its in-repeat reads on, for the `alts` field of the row (``meta.alts_field``).

    The tracts of the row's motif, less those that overlap the locus' own read window (its tract +- ALT_SPAN bases on
    its contig: those reads are fetched already), merged on a contig while the gap to the next tract is less than
    `read_length` (a read must not be fetched twice); the `max_alts` regions with the longest tracts are kept (ties:
    FASTA contig order, then start).  -> the kept regions in (contig, start) order as ``contig:start-end`` (0-based,
    end exclusive, how ``tred.alt_regions`` hands them to the fetch) joined by '|'; empty when none qualifies."""
    from .fasta import canonical_code
    from .meta import REF, get_region, location_field
    contig, first, last = get_region(locus_row[location_field(ref or REF)])
    motif = locus_row["motif"]
    names, t = tracts["contigs"], tracts["tracts"]
    t = t[(t["period"] == len(motif)) & (t["code"] == canonical_code(motif))]
    lo, hi = first - 1 - ALT_SPAN, last + ALT_SPAN
    regions = []                                        # [contig index, start, end, longest tract]
    for c, s, n in zip(t["contig"].tolist(), t["start"].tolist(), t["length"].tolist()):
        if names[c] == contig and s < hi and s + n > lo:
            continue
        if regions and regions[-1][0] == c and s - regions[-1][2] < read_length:
            regions[-1][2] = max(regions[-1][2], s + n)
            regions[-1][3] = max(regions[-1][3], n)
        else:
            regions.append([c, s, s + n, n])
    kept = sorted(regions, key=lambda r: (-r[3], r[0], r[1]))[:max_alts]
    return "|".join("{}:{}-{}".format(names[c], s, e) for c, s, e, _ in sorted(kept))


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m tredparse_b200.strprofile",
                                 description="STR profiles of whole BAMs (in-repeat reads found on the GPU) and their "
                                             "cohort comparison")
    sub = ap.add_subparsers(dest="cmd", required=True)
    pp = sub.add_parser("profile", help="one <sample>.str_profile.json per BAM (samples one after another, one GPU)")
    pp.add_argument("bams", nargs="+", help="BAM files (an index is not needed); '-' reads one BAM from stdin")
    pp.add_argument("--workdir", default=".")
    pp.add_argument("--min-period", type=int, default=2)
    pp.add_argument("--max-period", type=int, default=20)
    pp.add_argument("--purity-num", type=int, default=9)
    pp.add_argument("--purity-den", type=int, default=10)
    pp.add_argument("--min-read-len", type=int, default=50)
    pp.add_argument("--min-anchor-mapq", type=int, default=MIN_ANCHOR_MAPQ)
    pp.add_argument("--merge-distance", type=int, default=MERGE_DISTANCE)
    pp.add_argument("--slab-bytes", type=int, default=0, help="compressed bytes read per step (0: 128 MiB)")
    po = sub.add_parser("outliers", help="rank the samples of a cohort by region and motif")
    po.add_argument("profiles", nargs="+", help="<sample>.str_profile.json files")
    po.add_argument("--tsv", default=None, help="output table (default: stdout)")
    po.add_argument("--merge-distance", type=int, default=None)
    pl = sub.add_parser("loci", help="a sites JSON of the loci behind the outlier regions, for tred.py --tred NAME",
                        description="Build a locus from the reference at every outlier region with z >= --min-z and "
                                    "write them as one sites JSON. Genotype them with python -m tredparse_b200.tred "
                                    "samples.csv --tred NAME ... run from the directory that holds sites/ (indexed "
                                    "or unindexed BAMs, one or more GPUs). A BAM streamed through a pipe or stdin "
                                    "has to be streamed again to genotype the discovered loci; `python -m "
                                    "tredparse_b200.tred - --str-profile` gives its catalogue calls and its profile "
                                    "from one read.")
    pl.add_argument("tsv", help="the table `outliers` wrote")
    pl.add_argument("--fasta", required=True, help="the reference the BAMs are aligned to, plain text or bgzipped "
                                                   "(bgzip, not plain gzip); its .fai is used when present")
    pl.add_argument("--profiles", nargs="+", required=True,
                    help="<sample>.str_profile.json files: the read length is the largest among them")
    pl.add_argument("--min-z", type=float, default=3.0)
    pl.add_argument("--ref", default="hg38", choices=("hg38", "hg38_nochr", "hg19", "hg19_nochr"),
                    help="the tred.py --ref the loci are for (selects the location field)")
    pl.add_argument("--window", type=int, default=LOCUS_WINDOW, help="bases searched either side of a region")
    pl.add_argument("--min-ref-units", type=int, default=MIN_REF_UNITS)
    pl.add_argument("--out", default=os.path.join("sites", "discovered.json"))
    pl.add_argument("--alts", action="store_true",
                    help="give every locus the reference's other tracts of its motif as alt regions, where an aligner "
                         "may have placed its in-repeat reads (one GPU scan of the FASTA)")
    pl.add_argument("--max-alts", type=int, default=MAX_ALTS, help="alt regions kept per locus (longest tracts first)")
    pl.add_argument("--min-alt-len", type=int, default=MIN_TRACT_LEN,
                    help="bases an alt tract needs (default: BWA-MEM's minimum alignment score)")
    pl.add_argument("--max-interruption", type=int, default=0,
                    help="join tracts of one motif across interruptions of up to this many bases (0 to 20; 0: pure "
                         "tracts only), for the locus tract and --alts, when the joined tract is as pure as an "
                         "in-repeat read: the purity is the profiles' (DESIGN §4.5.1)")
    a = ap.parse_args(argv)
    if a.cmd == "loci":
        from .fasta import Fasta
        with open(a.tsv) as fp:
            rows = read_tsv(fp)
        read_length, purities = 0, set()
        for f in a.profiles:
            with open(f) as fp:
                prof = json.load(fp)
            read_length = max(read_length, int(prof["read_length"]))
            prm = prof.get("params", {})
            purities.add((prm.get("purity_num"), prm.get("purity_den")))
        if read_length <= 0:
            ap.error("the profiles give no read length")
        if not 0 <= a.max_interruption <= 20:
            ap.error("--max-interruption must be 0 to 20 (got {})".format(a.max_interruption))
        purity = (9, 10)
        if a.max_interruption:                          # the in-repeat reads' purity, one for the cohort
            if len(purities) != 1 or None in next(iter(purities)):
                ap.error("--max-interruption needs one purity (params.purity_num / purity_den) in every profile; "
                         "they give {}".format(sorted(purities, key=str)))
            purity = next(iter(purities))
        try:
            fasta = Fasta(a.fasta)
        except (IOError, ValueError) as e:
            ap.error(str(e))
        sites, skipped = discover_loci(rows, fasta, read_length, a.min_z, a.window, a.min_ref_units, a.ref,
                                       a.max_interruption, purity)
        below = sum(1 for r in rows if r["z"] < a.min_z)
        for r, why in skipped:
            where = r["contig"] if r["start"] is None else "{}:{}-{}".format(r["contig"], r["start"], r["end"])
            print("skipped {} {} (z {:.4f}): {}".format(where, r["motif"], r["z"], why), file=sys.stderr)
        print("{} rows below --min-z {}".format(below, a.min_z), file=sys.stderr)
        if a.alts and sites:
            from .meta import alts_field
            try:
                tracts = fasta.tracts({row["motif"] for row in sites.values()}, min_len=a.min_alt_len,
                                      max_interrupt=a.max_interruption, purity=purity)
            except _lib.TredswError as e:
                ap.exit(1, "loci --alts: {}\n".format(e))
            for name, row in sites.items():
                row[alts_field(a.ref)] = alt_regions_for(row, tracts, read_length, a.max_alts, a.ref)
                n = len(row[alts_field(a.ref)].split("|")) if row[alts_field(a.ref)] else 0
                print("{}: {} alt regions".format(name, n), file=sys.stderr)
        if os.path.dirname(a.out):
            os.makedirs(os.path.dirname(a.out), exist_ok=True)
        with open(a.out, "w") as fp:
            json.dump(sites, fp, indent=1, sort_keys=True)
            fp.write("\n")
        for name in sites:
            print(name)
        return 0
    if a.cmd == "profile":
        # one file per sample key: keys that repeat would overwrite each other (stdin's key is known once it is open)
        keys = [sample_key(b, None) for b in a.bams if b != "-"]
        if len(set(keys)) != len(keys) or a.bams.count("-") > 1:
            ap.error("sample keys repeat among the inputs: {}".format(sorted(k for k in set(keys) if keys.count(k) > 1) or "-"))
        os.makedirs(a.workdir, exist_ok=True)
        written = set()
        for bam in a.bams:
            prof = profile(bam, min_period=a.min_period, max_period=a.max_period, purity_num=a.purity_num,
                           purity_den=a.purity_den, min_read_len=a.min_read_len, min_anchor_mapq=a.min_anchor_mapq,
                           merge_distance=a.merge_distance, slab_bytes=a.slab_bytes or None)
            if prof["sample"] in written:
                ap.error("{}: its sample key `{}` is that of another input".format(bam, prof["sample"]))
            written.add(prof["sample"])
            out = os.path.join(a.workdir, "{}.str_profile.json".format(prof["sample"]))
            write_profile(prof, out)
            print(out)
        return 0
    profs = []
    for f in a.profiles:
        with open(f) as fp:
            profs.append(json.load(fp))
    rows = outliers(profs, merge_distance=a.merge_distance)
    samples = [p["sample"] for p in profs]
    if a.tsv:
        with open(a.tsv, "w") as fp:
            write_tsv(rows, samples, fp)
    else:
        write_tsv(rows, samples, sys.stdout)
    return 0


if __name__ == "__main__":
    sys.exit(main())
