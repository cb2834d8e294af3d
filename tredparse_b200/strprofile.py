"""
STR profile of a whole BAM: the in-repeat reads (IRRs, reads made almost entirely of one short motif) of every record,
found on the GPU in one streaming scan of the file (``ingest.scan_sample(..., irr=IrrParams())``, DESIGN §4.5),
anchored by their mapped mates and merged into regions per motif; then a cohort comparison that ranks the samples
with more anchored IRRs in a region than the rest of the cohort — expansions outside the catalogue.

    prof = strprofile.profile("x.bam")                 # or "-" / a FIFO: read once, in order
    rows = strprofile.outliers([prof_a, prof_b, ...])  # highest z first

    python -m tredparse_b200.strprofile profile x.bam [y.bam ... | -] --workdir w
    python -m tredparse_b200.strprofile outliers w/*.str_profile.json --tsv out.tsv
    python -m tredparse_b200.strprofile loci out.tsv --fasta ref.fa --profiles w/*.str_profile.json
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
from .ingest import BamIngest, IrrParams, is_stream, scan_sample

MIN_ANCHOR_MAPQ = 50
MERGE_DISTANCE = 500
NORM_DEPTH = 40.0
LOCUS_WINDOW = 1000
MIN_REF_UNITS = 3
LOCUS_FLANK = 18
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


def locus_for(row, fasta, read_length, window=LOCUS_WINDOW, min_ref_units=MIN_REF_UNITS, ref=None):
    """The locus behind a region row of ``outliers`` -> (name, locus row for ``meta.TRED``); raises Skip(reason).

    Candidate units are the k rotations of the row's canonical motif (period k) and the k rotations of its reverse
    complement.  The tract is the longest run of exact, back-to-back copies of one candidate unit in the reference
    window [start - window, end + window) clipped to the contig: the region spans the anchors, mates that lie up to a
    fragment from the tract.  Ties go to the run whose centre is closest to the region's centre, then to the leftmost
    run.  Reasons to skip: ``no position`` (a motif-only row), ``contig not in FASTA``, ``no reference tract`` (fewer
    than `min_ref_units` copies), ``flank outside contig``, ``N in flank`` (any base but A, C, G, T in the 18 bases
    either side).

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
    # copies[i]: back-to-back copies of the candidate unit seq[i:i+k] from i on (right to left: one pass)
    copies = [0] * (len(seq) + k)
    for i in range(len(seq) - k, -1, -1):
        u = seq[i:i + k]
        if u in units:
            copies[i] = 1 + (copies[i + k] if seq[i + k:i + 2 * k] == u else 0)
    centre2 = row["start"] + row["end"] - 2 * lo         # twice the region's centre, in window coordinates
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


def discover_loci(rows, fasta, read_length, min_z=3.0, window=LOCUS_WINDOW, min_ref_units=MIN_REF_UNITS, ref=None):
    """The loci of the outlier rows with z >= min_z, in row order -> ({name: locus row}, [(row, reason)] of the rows
    skipped).  Rows that resolve to one (contig, first base, repeat) — the left and right anchors of a long expansion
    can make two regions — give one locus, the first row's."""
    sites, skipped = {}, []
    for row in rows:
        if row["z"] < min_z:
            continue
        try:
            name, locus = locus_for(row, fasta, read_length, window, min_ref_units, ref)
        except Skip as e:
            skipped.append((row, str(e)))
            continue
        sites.setdefault(name, locus)
    return sites, skipped


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
                                    "was read once by `profile`: genotyping needs it streamed again.")
    pl.add_argument("tsv", help="the table `outliers` wrote")
    pl.add_argument("--fasta", required=True, help="the reference the BAMs are aligned to (plain text; its .fai is "
                                                   "used when present)")
    pl.add_argument("--profiles", nargs="+", required=True,
                    help="<sample>.str_profile.json files: the read length is the largest among them")
    pl.add_argument("--min-z", type=float, default=3.0)
    pl.add_argument("--ref", default="hg38", choices=("hg38", "hg38_nochr", "hg19", "hg19_nochr"),
                    help="the tred.py --ref the loci are for (selects the location field)")
    pl.add_argument("--window", type=int, default=LOCUS_WINDOW, help="bases searched either side of a region")
    pl.add_argument("--min-ref-units", type=int, default=MIN_REF_UNITS)
    pl.add_argument("--out", default=os.path.join("sites", "discovered.json"))
    a = ap.parse_args(argv)
    if a.cmd == "loci":
        from .fasta import Fasta
        with open(a.tsv) as fp:
            rows = read_tsv(fp)
        read_length = 0
        for f in a.profiles:
            with open(f) as fp:
                read_length = max(read_length, int(json.load(fp)["read_length"]))
        if read_length <= 0:
            ap.error("the profiles give no read length")
        try:
            fasta = Fasta(a.fasta)
        except (IOError, ValueError) as e:
            ap.error(str(e))
        sites, skipped = discover_loci(rows, fasta, read_length, a.min_z, a.window, a.min_ref_units, a.ref)
        below = sum(1 for r in rows if r["z"] < a.min_z)
        for r, why in skipped:
            where = r["contig"] if r["start"] is None else "{}:{}-{}".format(r["contig"], r["start"], r["end"])
            print("skipped {} {} (z {:.4f}): {}".format(where, r["motif"], r["z"], why), file=sys.stderr)
        print("{} rows below --min-z {}".format(below, a.min_z), file=sys.stderr)
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
            with open(out, "w") as fp:
                json.dump(prof, fp, indent=1, sort_keys=True)
                fp.write("\n")
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
