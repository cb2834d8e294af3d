"""
TRED catalogue: the loci, their flanks / motif / cut-offs and alternative regions.

Mirrors ``tredparse/meta.py`` (``TREDsRepo`` :29-100, ``TRED`` :103-140, ``get_region`` :143-150) on top
of the compact tables in ``tredparse_b200/data`` (derived by ``tools/make_data.py``); user loci are
picked up from ``<sites>/*.json`` exactly like ``meta.py:44-49``.  No pandas: rows are plain dicts.
"""
import csv
import json
import os.path as op
from glob import glob

from .utils import datafile

REF = "hg38"
SITES = "sites"


def get_region(location):
    """'chr4:3074877-3074933' -> ('chr4', 3074877, 3074933)"""
    chr, location = location.split(":")
    start, end = location.split("-")
    return chr, int(start), int(end)


def location_field(ref=REF):
    """the row field that holds a locus' location on reference `ref` (hg38: repeat_location, hg19:
    repeat_location.hg19; the _nochr variants use the field of their build)"""
    return "repeat_location" if ref == REF else "repeat_location." + ref.split("_")[0]


def alts_field(ref=REF):
    """the field that holds a locus' alt regions on reference `ref`, in alts.tsv and in a user row (hg38: alts, hg19:
    alts.hg19; the _nochr variants use the field of their build): `contig:start-end` regions (0-based, end exclusive)
    joined by '|', empty for none"""
    return "alts" if ref == REF else "alts." + ref.split("_")[0]


def parse_alts(value):
    """an alts field -> [(contig, start, end)]"""
    return [get_region(x) for x in value.split("|")] if value.strip() else []


def locus_names(sites=SITES):
    """the names of the catalogue loci and of the user loci in <sites>/*.json, in TREDsRepo's order, without reading
    their rows (a user locus may carry the location of one reference build only)"""
    with open(datafile("loci.tsv")) as fp:
        names = [row["name"] for row in csv.DictReader(fp, delimiter="\t")]
    for s in sorted(glob("{}/*.json".format(sites))):
        with open(s) as fp:
            names += [str(name) for name in json.load(fp)]
    return names


def _num(x):
    try:
        f = float(x)
    except (TypeError, ValueError):
        return x
    return int(f) if f == int(f) else f


class TRED(object):
    def __init__(self, name, row, ref=REF, alt=()):
        self.row = row
        self.name = name
        self.alt = list(alt)
        self.repeat = row["repeat"]
        location = row[location_field(ref)]
        if "_nochr" in ref:
            location = location.replace("chr", "")
        self.chr, self.repeat_start, self.repeat_end = get_region(location)
        self.ref_copy = (self.repeat_end - self.repeat_start + 1) // len(self.repeat)
        self.prefix = row["prefix"]
        self.suffix = row["suffix"]
        self.cutoff_prerisk = _num(row["cutoff_prerisk"])
        self.cutoff_risk = _num(row["cutoff_risk"])
        self.inheritance = row["inheritance"]
        self.is_xlinked = self.inheritance[0] == "X"
        self.is_recessive = self.inheritance[-1] == "R"
        self.is_expansion = row["mutation_nature"] == "increase"
        self.ploidy = 2

    @property
    def allele_freq(self):
        """{units: count} parsed from the catalogue's '{5:8667,6:59,...}' column (cohort simulator)."""
        s = (self.row.get("allele_freq") or "").strip().strip("{}")
        out = {}
        for kv in s.split(","):
            if ":" in kv:
                k, v = kv.split(":")
                out[int(k)] = int(v)
        return out

    def __repr__(self):
        return "{} inheritance={} id={}_{}_{}".format(self.name, self.inheritance, self.chr,
                                                      self.repeat_start, self.repeat)

    def __str__(self):
        return ";".join(str(x) for x in (self.name, self.repeat, self.chr, self.repeat_start,
                                         self.repeat_end, self.prefix, self.suffix))


class TREDsRepo(dict):
    def __init__(self, ref=REF, toy=False, sites=SITES):
        self.ref = ref
        alts = self.get_alts(ref)
        self.names = []
        self.rows = {}
        with open(datafile("loci.tsv")) as fp:
            for row in csv.DictReader(fp, delimiter="\t"):
                name = row.pop("name")
                self[name] = TRED(name, row, ref=ref, alt=alts.get(name, []))
                self.rows[name] = row
                self.names.append(name)
        for s in sorted(glob("{}/*.json".format(sites))):
            with open(s) as fp:
                for name, row in json.load(fp).items():
                    name = str(name)
                    alt = parse_alts(row[alts_field(ref)]) if alts_field(ref) in row else alts.get(name, [])
                    self[name] = TRED(name, row, ref=ref, alt=alt)
                    self.rows[name] = row
                    self.names.append(name)
        if toy:
            tr = self.get("HD")
            tr.name = "toy"
            tr.chr = "CHR4"
            tr.repeat_start = 1001
            tr.repeat_end = 1057
            self[tr.name] = tr

    def set_ploidy(self, haploid):
        if not haploid:
            return
        for v in self.values():
            if v.chr in haploid:
                v.ploidy = 1

    def get_info(self, tredName):
        tr = self.get(tredName)
        info = "END={};MOTIF={};NS=1;REF={};CR={};IH={};RL={};VT=STR".format(
            tr.repeat_end, tr.repeat, tr.ref_copy, tr.cutoff_risk, tr.inheritance,
            tr.ref_copy * len(tr.repeat))
        return tr.chr, tr.repeat_start, tr.ref_copy, tr.repeat, info

    @staticmethod
    def get_alts(ref):
        field = alts_field(ref)
        alts = {}
        with open(datafile("alts.tsv")) as fp:
            for row in csv.DictReader(fp, delimiter="\t"):
                alts[row["name"]] = parse_alts(row.get(field) or "")
        return alts
