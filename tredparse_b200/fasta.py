"""
Random access to a plain-text FASTA file, as `samtools faidx` gives it.

    fa = Fasta("ref.fa")                  # uses ref.fa.fai when it exists, else indexes the file in memory
    fa.fetch("chr4", 3074876, 3074933)    # 0-based, half-open; uppercase bases
    fa.lengths()                          # {contig: length}

The index is the `.fai` format: per record its name (the header up to the first white space), length, the byte
offset of its first base, and the bases and bytes of each line.  Lines of any width work as long as every line of a
record but the last has the same width, which is what `samtools faidx` requires too.  An index built here stays in
memory: nothing is written next to the user's file.  Compressed files (gzip, BGZF) are refused.
"""
import os


class Fasta:
    def __init__(self, path):
        self.path = path
        with open(path, "rb") as fp:
            if fp.read(2) == b"\x1f\x8b":
                raise ValueError("{}: a compressed (gzip / BGZF) FASTA is not supported; decompress it first".format(path))
        fai = path + ".fai"
        self.index = self._read_fai(fai) if os.path.exists(fai) else self._build_index(path)

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
    def _build_index(path):
        """the .fai entries of `path`, from one pass over its lines"""
        index, name = {}, None
        length = offset = lb = lw = 0
        short = False                                   # a line shorter than the first was seen: it must be the last

        def close():
            if name is not None:
                index[name] = (length, offset, lb, lw)
        pos = 0
        with open(path, "rb") as fp:
            for line in fp:
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

    def fetch(self, contig, start, end):
        """the bases [start, end) of `contig` (0-based), uppercase, clipped to the contig; KeyError for a contig the
        file does not have"""
        if contig not in self.index:
            raise KeyError("contig `{}` is not in {}".format(contig, self.path))
        length, offset, lb, lw = self.index[contig]
        start, end = max(0, start), min(length, end)
        if end <= start:
            return ""
        first = offset + (start // lb) * lw + start % lb
        last = offset + ((end - 1) // lb) * lw + (end - 1) % lb
        with open(self.path, "rb") as fp:
            fp.seek(first)
            raw = fp.read(last - first + 1)
        seq = raw.replace(b"\n", b"").replace(b"\r", b"").decode("ascii").upper()
        if len(seq) != end - start:
            raise ValueError("{}: contig `{}` is shorter than its index says".format(self.path, contig))
        return seq
