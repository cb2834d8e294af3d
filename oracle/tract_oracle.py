"""
Plain-Python restatement of the reference tract scan (tredsw_ref_tracts, csrc/ref_tracts_device.cuh) and of the alt
regions of a discovered locus (strprofile.alt_regions_for), for the tests.  Nothing under tredparse_b200/ imports it.

Tract of period k: a maximal stretch [a, b) of bases in ACGTacgt (compared case-insensitively) with s[j] == s[j + k]
for every j in [a, b - k) gives [a, a + c k), c = (b - a) // k, unit s[a, a + k) upper-cased.  It is kept when the
unit's primitive root has period k, c >= min_units, c k >= min_len and the unit's canonical form is requested for k.
"""


def revcomp(s):
    return s.translate(str.maketrans("ACGT", "TGCA"))[::-1]


def canonical(unit):
    return min(m[i:] + m[:i] for m in (unit, revcomp(unit)) for i in range(len(unit)))


def code(motif):
    c = 0
    for b in motif:
        c = c * 4 + "ACGT".index(b)
    return c


def root_period(unit):
    k = len(unit)
    return next(e for e in range(1, k + 1) if k % e == 0 and all(unit[i] == unit[i - e] for i in range(e, k)))


def tracts(contigs, motifs, min_units=3, min_len=30):
    """contigs: {name: text of its bases} in FASTA order; motifs: strings.  -> [(contig index, start, length, period,
    canonical code)] by (contig, start, period)"""
    want = {(len(m), canonical(m.upper())) for m in motifs}
    out = []
    for ci, seq in enumerate(contigs.values()):
        s = seq.upper()
        n = len(s)
        ok = [ch in "ACGT" for ch in s]
        for k in sorted({k for k, _ in want}):
            a = 0
            while a < n:
                # the stretch from a: valid bases, each equal to the one k before it from a + k on
                b = a
                while b < n and ok[b] and (b < a + k or s[b] == s[b - k]):
                    b += 1
                c = (b - a) // k
                if c >= min_units and c * k >= min_len:
                    unit = s[a:a + k]
                    if root_period(unit) == k and (k, canonical(unit)) in want:
                        out.append((ci, a, c * k, k, code(canonical(unit))))
                # the next maximal stretch starts where this one's last k bases stop agreeing with it
                a = max(a + 1, b - k + 1) if b - a > k else a + 1
    return sorted(out, key=lambda t: (t[0], t[1], t[3]))


def alt_regions(tracts_, names, own, motif, read_length, max_alts=100, span=1000):
    """tracts_: tracts() output; names: contig names in FASTA order; own: (contig, first, last) of the locus (1-based,
    inclusive).  -> 'contig:start-end|...' as strprofile.alt_regions_for writes it"""
    k, cc = len(motif), code(canonical(motif))
    lo, hi = own[1] - 1 - span, own[2] + span
    regs = []
    for c, s, n, p, x in tracts_:
        if p != k or x != cc or (names[c] == own[0] and s < hi and s + n > lo):
            continue
        if regs and regs[-1][0] == c and s - regs[-1][2] < read_length:
            regs[-1] = [c, regs[-1][1], max(regs[-1][2], s + n), max(regs[-1][3], n)]
        else:
            regs.append([c, s, s + n, n])
    kept = sorted(regs, key=lambda r: (-r[3], r[0], r[1]))[:max_alts]
    return "|".join("{}:{}-{}".format(names[c], s, e) for c, s, e, _ in sorted(kept))
