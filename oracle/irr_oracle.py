"""
Oracle of the STR profile (tredparse_b200.strprofile, the IRR stage of the GPU scan): the definitions of DESIGN §4.5
restated in plain Python over bamio records — per-record classification of in-repeat reads (IRRs), the per-sample
profile (anchored and paired IRRs, regions of anchors) and the cohort outlier table.  Loops and dicts only: it shares
no code with the package beyond the BAM record reader.
"""
import math

from tredparse_b200 import bamio

DEFAULTS = dict(min_period=2, max_period=20, purity_num=9, purity_den=10, min_read_len=50)
SKIP = 0x100 | 0x200 | 0x400 | 0x800
_CODE = {"A": 0, "C": 1, "G": 2, "T": 3}


def classify(seq, min_period=2, max_period=20, purity_num=9, purity_den=10, min_read_len=50):
    """seq: a string of bases or a list of codes (0..3 = A C G T, anything else N) -> (period, motif bits); (0, 0)
    when the read is not an IRR"""
    codes = [_CODE.get(c, 4) for c in seq] if isinstance(seq, str) else [c if 0 <= c < 4 else 4 for c in seq]
    L = len(codes)
    if L < min_read_len:
        return 0, 0
    left = bytes(codes)                                    # N is 4 on the left, 5 on the right: never equal
    right = bytes(5 if c == 4 else c for c in codes)
    period = 0
    for k in range(min_period, max_period + 1):
        n = L - k
        m = sum(map(int.__eq__, left[:n], right[k:]))
        if m * purity_den >= purity_num * n:
            period = k
            break
    if not period:
        return 0, 0
    cons = []
    for j in range(period):
        cnt = [0, 0, 0, 0]
        for i in range(j, L, period):
            if codes[i] < 4:
                cnt[codes[i]] += 1
        best = 0
        for b in range(1, 4):
            if cnt[b] > cnt[best]:
                best = b
        cons.append(best)
    d = period
    for e in range(1, period):
        if period % e == 0 and all(cons[i] == cons[i % e] for i in range(period)):
            d = e
            break
    if d == 1:
        return 0, 0
    root = cons[:d]
    rc = [3 - b for b in reversed(root)]
    best = min(tuple(x[t:] + x[:t]) for x in (root, rc) for t in range(d))
    bits = 0
    for b in best:
        bits = bits * 4 + b
    return d, bits


def motif_string(period, bits):
    return "".join("ACGT"[(bits >> (2 * (period - 1 - i))) & 3] for i in range(period))


def record_mq(rec):
    """(MQ or None, the aux area could not be parsed); negative values read as 0"""
    try:
        v = rec.integer_tag("MQ")
    except ValueError:
        return None, True
    if v is None:
        return None, False
    return max(0, min(v, 2 ** 31 - 1)), False


def scan(path, params=None):
    """every record of the BAM -> dict(entries: the IRR records in file order, stats, references)"""
    p = dict(DEFAULTS, **(params or {}))
    sam = bamio.AlignmentFile(path)
    refs = list(zip(sam.references, sam.lengths))
    entries = []
    st = dict(records_considered=0, depth_bases=0, max_l_seq=0, unparsed_aux=0)
    for r in sam.fetch():
        if r.flag & SKIP:
            continue
        L = len(r.query_sequence)
        st["max_l_seq"] = max(st["max_l_seq"], L)
        if not r.flag & 4:
            st["depth_bases"] += L
        if L < p["min_read_len"]:
            continue
        st["records_considered"] += 1
        per, bits = classify(r.query_sequence, **p)
        if not per:
            continue
        mq, bad = record_mq(r)
        st["unparsed_aux"] += bad
        entries.append(dict(name=r.query_name, tid=r.reference_id, pos=r.reference_start, next_tid=r.next_reference_id,
                            next_pos=r.next_reference_start, flag=r.flag, mapq=r.mapping_quality,
                            mq=-1 if mq is None else mq, period=per, motif=bits))
    sam.close()
    st["irr_records"] = len(entries)
    return dict(entries=entries, stats=st, references=refs)


def join(entries):
    """the mate of every entry: the first entry of the same name with the other segment flag, -1 none"""
    seg = {}
    for k, e in enumerate(entries):
        f = e["flag"] & 0xC0
        if f in (0x40, 0x80):
            seg.setdefault(e["name"], {}).setdefault(f, k)
    mate = [-1] * len(entries)
    for d in seg.values():
        if 0x40 in d and 0x80 in d:
            mate[d[0x40]] = d[0x80]
            mate[d[0x80]] = d[0x40]
    return mate


def profile(path, params=None, min_anchor_mapq=50, merge_distance=500, sample=None):
    p = dict(DEFAULTS, **(params or {}))
    sc = scan(path, p)
    entries, refs = sc["entries"], sc["references"]
    mate = join(entries)
    motifs = {}
    st = dict(sc["stats"], anchors_without_mq=0, anchors_below_mapq=0, anchored_irrs=0, paired_irrs=0,
              irr_pairs_motif_mismatch=0)
    anchors = {}
    for k, e in enumerate(entries):
        key = motif_string(e["period"], e["motif"])
        if mate[k] >= 0:
            if e["flag"] & 0x40:
                o = entries[mate[k]]
                if (o["period"], o["motif"]) == (e["period"], e["motif"]):
                    motifs.setdefault(key, [0, 0])[1] += 1
                    st["paired_irrs"] += 1
                else:
                    st["irr_pairs_motif_mismatch"] += 1
            continue
        if not (e["flag"] & 1) or (e["flag"] & 8) or e["next_tid"] < 0:
            continue
        if e["mq"] < 0:
            st["anchors_without_mq"] += 1
        elif e["mq"] < min_anchor_mapq:
            st["anchors_below_mapq"] += 1
            continue
        motifs.setdefault(key, [0, 0])[0] += 1
        st["anchored_irrs"] += 1
        anchors.setdefault(key, []).append((e["next_tid"], e["next_pos"]))
    out = {}
    for key in sorted(motifs):
        regions = []
        for tid, pos in sorted(anchors.get(key, [])):
            if regions and regions[-1][0] == tid and pos - (regions[-1][2] - 1) <= merge_distance:
                regions[-1][2] = pos + 1
                regions[-1][3] += 1
            else:
                regions.append([tid, pos, pos + 1, 1])
        out[key] = {"anchored_irr_count": motifs[key][0], "paired_irr_count": motifs[key][1],
                    "regions": [{"contig": refs[t][0], "start": s, "end": e, "count": c} for t, s, e, c in regions]}
    total = sum(n for _, n in refs)
    params_out = dict(p, min_anchor_mapq=min_anchor_mapq, merge_distance=merge_distance)
    return {"sample": sample, "bam": path, "read_length": st["max_l_seq"],
            "depth": st["depth_bases"] / total if total else 0.0, "params": params_out, "stats": st, "profile": out}


def _z(xs, i):
    others = xs[:i] + xs[i + 1:]
    mean = sum(others) / len(others)
    sd = math.sqrt(sum((o - mean) ** 2 for o in others) / len(others))
    return (xs[i] - mean) / max(sd, 1.0)


def _row(contig, start, end, motif, samples, xs):
    zs = [_z(xs, i) for i in range(len(xs))]
    top = 0
    for i in range(1, len(zs)):
        if zs[i] > zs[top]:
            top = i
    return {"contig": contig, "start": start, "end": end, "motif": motif, "top_sample": samples[top], "z": zs[top],
            "counts": dict(zip(samples, xs))}


def outliers(profiles, merge_distance=None):
    if len(profiles) < 2:
        raise ValueError("a cohort needs at least two samples")
    md = profiles[0]["params"]["merge_distance"] if merge_distance is None else merge_distance
    samples = [p["sample"] for p in profiles]
    norm = [(40.0 / p["depth"]) if p["depth"] > 0 else 0.0 for p in profiles]
    rows = []
    motifs = sorted(set(m for p in profiles for m in p["profile"]))
    for motif in motifs:
        allr = sorted((r["contig"], r["start"], r["end"]) for p in profiles for r in p["profile"].get(motif, {}).get("regions", []))
        cohort = []
        for c, s, e in allr:
            if cohort and cohort[-1][0] == c and s - (cohort[-1][2] - 1) <= md:
                cohort[-1][2] = max(cohort[-1][2], e)
            else:
                cohort.append([c, s, e])
        for c, s, e in cohort:
            xs = []
            for p, f in zip(profiles, norm):
                n = sum(r["count"] for r in p["profile"].get(motif, {}).get("regions", [])
                        if r["contig"] == c and s <= r["start"] < e)
                xs.append(n * f)
            rows.append(_row(c, s, e, motif, samples, xs))
        xs = [p["profile"].get(motif, {}).get("paired_irr_count", 0) * f for p, f in zip(profiles, norm)]
        rows.append(_row("-", None, None, motif, samples, xs))
    rows.sort(key=lambda r: (-r["z"], r["motif"], r["contig"], -1 if r["start"] is None else r["start"]))
    return rows
