"""
Random access to a FASTA file, plain text or bgzipped (BGZF), as `samtools faidx` gives it.

    fa = Fasta("ref.fa")                  # uses ref.fa.fai when it exists, else indexes the file in memory
    fa = Fasta("ref.fa.gz")               # the same for `bgzip ref.fa` (its .fai, not its .gzi)
    fa.fetch("chr4", 3074876, 3074933)    # 0-based, half-open; uppercase bases
    fa.lengths()                          # {contig: length}
    fa.tracts(["AAGGG", "AGC"])           # every tract of these motifs, found by one GPU scan of the file

The index is the `.fai` format: per record its name (the header up to the first white space), length, the byte
offset of its first base, and the bases and bytes of each line.  Lines of any width work as long as every line of a
record but the last has the same width, which is what `samtools faidx` requires too.  An index built here stays in
memory: nothing is written next to the user's file.

A BGZF file is recognised by its first block (gzip magic, FEXTRA, a `BC` subfield); its `.fai` offsets are offsets
into the inflated text, as `samtools faidx` writes them.  `fetch` inflates only the blocks a window touches (found by
one walk of the block headers, with every block's length and CRC-32 checked), and `tracts` inflates the blocks on the
GPU.  Without a `.fai` the index is built by inflating the whole file on the host, which for a whole genome takes
minutes: run `samtools faidx ref.fa.gz` once instead.  A plain gzip file cannot be read by block and is refused.
"""
import bisect
import gzip
import os
import struct
import zlib

import numpy as np

from . import bamio

MIN_REF_UNITS = 3       # copies a reference tract needs (strprofile.locus_for uses the same)
MIN_TRACT_LEN = 30      # bases a tract needs: BWA-MEM's default minimum alignment score


def canonical_code(motif):
    """the canonical code of a motif: the smallest rotation of it and of its reverse complement, 2 bits a base
    (A C G T = 0 1 2 3), first base most significant — the code of tredsw_irr_entry.motif and tredsw_tract.code"""
    motif = motif.upper()
    rc = motif.translate(str.maketrans("ACGT", "TGCA"))[::-1]
    best = min(m[i:] + m[:i] for m in (motif, rc) for i in range(len(motif)))
    code = 0
    for b in best:
        code = code * 4 + "ACGT".index(b)
    return code


def _is_bgzf(fp):
    """the file's first block is BGZF: gzip magic, FEXTRA and a `BC` subfield"""
    head = fp.read(12)
    if len(head) < 12 or head[:2] != b"\x1f\x8b" or not head[3] & 4:
        return False
    extra = fp.read(struct.unpack_from("<H", head, 10)[0])
    off = 0
    while off + 4 <= len(extra):
        si1, si2, slen = struct.unpack_from("<BBH", extra, off)
        if (si1, si2, slen) == (66, 67, 2):
            return True
        off += 4 + slen
    return False


class Fasta:
    def __init__(self, path):
        self.path = path
        self.blocks = None               # BGZF: (compressed offset, inflated offset, inflated size) of every block
        with open(path, "rb") as fp:
            if fp.read(2) == b"\x1f\x8b":
                fp.seek(0)
                if not _is_bgzf(fp):
                    raise ValueError("{}: a compressed FASTA that is not BGZF (plain gzip) is not supported; recompress "
                                     "it with `bgzip`".format(path))
                self.blocks = bamio.bgzf_blocks(path)
                self._block_starts = [b[1] for b in self.blocks]
        fai = path + ".fai"
        if os.path.exists(fai):
            self.index = self._read_fai(fai)
        elif self.blocks is None:
            with open(path, "rb") as lines:
                self.index = self._build_index(path, lines)
        else:
            try:
                with gzip.open(path, "rb") as lines:
                    self.index = self._build_index(path, lines)
            except (zlib.error, EOFError, gzip.BadGzipFile) as e:
                raise IOError("{}: corrupt BGZF data: {}".format(path, e))

    @staticmethod
    def _read_fai(fai):
        index = {}
        with open(fai) as fp:
            for line in fp:
                if line.strip():
                    name, length, offset, lb, lw = line.rstrip("\n").split("\t")[:5]
                    index[name] = (int(length), int(offset), int(lb), int(lw))
        return index

    @staticmethod
    def _build_index(path, lines):
        """the .fai entries of `path`, from one pass over `lines`, its (inflated) text line by line"""
        index, name = {}, None
        length = offset = lb = lw = 0
        short = False                                   # a line shorter than the first was seen: it must be the last

        def close():
            if name is not None:
                index[name] = (length, offset, lb, lw)
        pos = 0
        for line in lines:
            if line.startswith(b">"):
                close()
                name = line[1:].split()[0].decode() if line[1:].split() else ""
                if name in index:
                    raise ValueError("{}: contig `{}` occurs twice".format(path, name))
                length, offset, lb, lw, short = 0, pos + len(line), 0, 0, False
            elif name is not None:
                bases = len(line.rstrip(b"\r\n"))
                if bases:
                    wider = lb and (bases > lb or (line.endswith(b"\n") and len(line) - bases != lw - lb))
                    if short or wider:
                        raise ValueError("{}: lines of unequal width in contig `{}`".format(path, name))
                    if not lb:
                        lb, lw = bases, len(line)
                    short = bases < lb
                    length += bases
                elif length:
                    short = True                   # an empty line ends the record's sequence
            pos += len(line)
        close()
        return index

    def __contains__(self, contig):
        return contig in self.index

    def lengths(self):
        return {name: e[0] for name, e in self.index.items()}

    def tracts(self, motifs, min_units=MIN_REF_UNITS, min_len=MIN_TRACT_LEN, step_bytes=0, ctx=None, emulate=False,
               max_interrupt=0, purity=(9, 10)):
        """Every tract of the motifs (strings of 2 to 20 bases; a motif stands for all its rotations on both strands)
        in the whole file, from one scan on the GPU (``_lib.ref_tracts``, DESIGN §4.5; a BGZF file is inflated
        there block by block): a maximal stretch of exact
        back-to-back copies of a unit whose primitive root has the motif's length, at least `min_units` copies and
        `min_len` bases long, lowercase bases equal to uppercase, anything but ACGT breaking it.  -> dict(contigs:
        the contig names in FASTA order, tracts: a ``_lib.TRACT_DTYPE`` array by (contig, start, period) with contig
        an index into contigs, start 0-based, length a whole number of units, code the canonical code; stats: steps,
        bytes, bases, invalid_bases, tracts, per-step host read and device ms, and comp_bytes and blocks, the
        compressed bytes read and blocks inflated, 0 for a text file; segments: per tract, the segments of its chain,
        an int32 array).  ``max_interrupt`` >= 1 (at most 20) also joins tracts of one motif across interruptions of
        up to that many bases when the joined tract has `purity` (num, den) (DESIGN §4.5.1); 0 is the pure rule.
        ``ctx``: a ``_lib.Context``; ``emulate``: the serial host emulation of the device code (test infrastructure
        only)."""
        from . import _lib
        names = list(self.index)
        contigs = np.array([self.index[n] for n in names], dtype=np.int64).reshape(-1, 4)
        fai = np.zeros(len(names), dtype=_lib.FAI_ENTRY_DTYPE)
        for f, col in zip(("length", "offset", "line_bases", "line_width"), contigs.T):
            fai[f] = col
        motifs = sorted({(len(m), canonical_code(m)) for m in motifs})
        tracts, stats = _lib.ref_tracts(self.path, fai, motifs, min_units, min_len, step_bytes, ctx=ctx, emulate=emulate,
                                        max_interrupt=max_interrupt, purity_num=purity[0], purity_den=purity[1])
        return {"contigs": names, "tracts": tracts, "stats": stats, "segments": stats["segments"]}

    def fetch(self, contig, start, end):
        """the bases [start, end) of `contig` (0-based), uppercase, clipped to the contig; KeyError for a contig the
        file does not have; IOError for a corrupt BGZF block among those the window touches"""
        if contig not in self.index:
            raise KeyError("contig `{}` is not in {}".format(contig, self.path))
        length, offset, lb, lw = self.index[contig]
        start, end = max(0, start), min(length, end)
        if end <= start:
            return ""
        first = offset + (start // lb) * lw + start % lb
        last = offset + ((end - 1) // lb) * lw + (end - 1) % lb
        if self.blocks is None:
            with open(self.path, "rb") as fp:
                fp.seek(first)
                raw = fp.read(last - first + 1)
        else:
            raw = self._read_inflated(first, last - first + 1)
        seq = raw.replace(b"\n", b"").replace(b"\r", b"").decode("ascii").upper()
        if len(seq) != end - start:
            raise ValueError("{}: contig `{}` is shorter than its index says".format(self.path, contig))
        return seq

    def _read_inflated(self, at, n):
        """n bytes of a BGZF file's inflated text from inflated offset `at` (fewer at the end of the file): the blocks
        from the one holding `at` on, each checked for length and CRC-32"""
        b = bisect.bisect_right(self._block_starts, at) - 1
        coff, uoff, isize = self.blocks[b]
        if at >= uoff + isize:                          # past the inflated end
            return b""
        reader = bamio.BGZFReader(self.path)
        try:
            reader.seek((coff << 16) | (at - uoff))
            return reader.read(n)
        except zlib.error as e:
            raise IOError("{}: corrupt BGZF block at or after offset {}: {}".format(self.path, coff, e))
        finally:
            reader.close()
