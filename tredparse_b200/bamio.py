"""
Dependency-free BAM / BGZF / BAI reader and a minimal BAM writer (host glue).

The reference reads BAMs through pysam (``tredparse/bam_parser.py:22,432-436``); pysam / htslib are
not available to this build, and the hot path only needs four things from a BAM, all provided here
with pysam's semantics:

* ``AlignmentFile.fetch(chr, start, end)``  — records overlapping the 0-based half-open window, in
  file order, located through the ``.bai`` index when present (``bam_parser.py:206,226,333``);
* the per-record attributes the reference touches (``query_sequence``, ``query_name``,
  ``is_unmapped``, ``reference_start``, ``reference_end``, ``next_reference_id``,
  ``next_reference_start``, ``is_paired``, ``is_duplicate``, ``is_reverse``, ``query_length``,
  ``query_alignment_start``, ``query_alignment_end``);
* ``pileup``-style mean depth (``bam_parser.py:404-411``) — see :func:`region_depth`;
* ``fetch()`` without a region for read-length detection (``bam_parser.py:381-391``).

The writer exists so that synthetic cohorts and the trimmed test fixtures can go through the very same
``BamParser`` entry point as real data.
"""
from __future__ import annotations

import struct
import zlib
import os
from typing import Iterator, List, Optional, Tuple

import numpy as np

_SEQ_DECODE = "=ACMGRSVTWYHKDBN"
_CIGAR_OPS = "MIDNSHP=X"
# consumes (query, reference) per op code
_CONSUMES_Q = (1, 1, 0, 0, 1, 0, 0, 1, 1)
_CONSUMES_R = (1, 0, 1, 1, 0, 0, 0, 1, 1)

_NIB2 = np.array([a + b for a in _SEQ_DECODE for b in _SEQ_DECODE])

FUNMAP, FPAIRED, FREVERSE, FSECONDARY, FQCFAIL, FDUP = 0x4, 0x1, 0x10, 0x100, 0x200, 0x400


class AlignedSegment:
    """The slice of pysam.AlignedSegment the reference uses."""

    __slots__ = ("query_name", "flag", "reference_id", "reference_start", "mapping_quality",
                 "cigartuples", "next_reference_id", "next_reference_start", "template_length",
                 "query_sequence", "_qual", "_ref_end", "aux")

    def __init__(self, query_name, flag, reference_id, reference_start, mapping_quality, cigartuples,
                 next_reference_id, next_reference_start, template_length, query_sequence, qual=None, aux=b""):
        self.query_name = query_name
        self.flag = flag
        self.reference_id = reference_id
        self.reference_start = reference_start
        self.mapping_quality = mapping_quality
        self.cigartuples = cigartuples
        self.next_reference_id = next_reference_id
        self.next_reference_start = next_reference_start
        self.template_length = template_length
        self.query_sequence = query_sequence
        self._qual = qual
        self._ref_end = None
        self.aux = aux          # the raw optional fields (tag, type, value ...) as stored in the record

    # flags -------------------------------------------------------------------------------------
    @property
    def is_unmapped(self): return bool(self.flag & FUNMAP)
    @property
    def is_paired(self): return bool(self.flag & FPAIRED)
    @property
    def is_reverse(self): return bool(self.flag & FREVERSE)
    @property
    def is_duplicate(self): return bool(self.flag & FDUP)
    @property
    def is_secondary(self): return bool(self.flag & FSECONDARY)
    @property
    def is_qcfail(self): return bool(self.flag & FQCFAIL)

    # optional fields -----------------------------------------------------------------------------
    def integer_tag(self, tag):
        """The value of the first field `tag` of an integer type (c C s S i I) in the raw aux bytes, None when there is
        none (fields of the types A Z H B f are skipped).  Raises ValueError when the aux area cannot be parsed."""
        a, data, want = 0, self.aux, tag.encode("latin-1")
        sizes = {b"A": 1, b"c": 1, b"C": 1, b"s": 2, b"S": 2, b"i": 4, b"I": 4, b"f": 4}
        ints = {b"c": "<b", b"C": "<B", b"s": "<h", b"S": "<H", b"i": "<i", b"I": "<I"}
        while a < len(data):
            if a + 3 > len(data):
                raise ValueError("truncated aux field")
            t = data[a + 2:a + 3]
            hit = data[a:a + 2] == want
            a += 3
            if t in sizes:
                if a + sizes[t] > len(data):
                    raise ValueError("truncated aux field")
                if hit and t in ints:
                    return struct.unpack_from(ints[t], data, a)[0]
                a += sizes[t]
            elif t in (b"Z", b"H"):
                end = data.find(b"\0", a)
                if end < 0:
                    raise ValueError("unterminated aux string")
                a = end + 1
            elif t == b"B":
                if a + 5 > len(data):
                    raise ValueError("truncated aux array")
                sub = data[a:a + 1]
                (n,) = struct.unpack_from("<I", data, a + 1)
                if sub not in sizes or sub == b"A" or a + 5 + n * sizes[sub] > len(data):
                    raise ValueError("bad aux array")
                a += 5 + n * sizes[sub]
            else:
                raise ValueError("unknown aux type {!r}".format(t))
        return None

    # geometry ----------------------------------------------------------------------------------
    @property
    def query_length(self):
        return len(self.query_sequence)

    @property
    def reference_length(self):
        return sum(l for op, l in self.cigartuples if _CONSUMES_R[op])

    @property
    def reference_end(self):
        """0-based exclusive end on the reference; None for records without an alignment
        (pysam returns None as well)."""
        if self._ref_end is None:
            if self.is_unmapped or not self.cigartuples:
                return None
            self._ref_end = self.reference_start + self.reference_length
        return self._ref_end

    @property
    def query_alignment_start(self):
        """Offset of the first aligned base in query_sequence (soft clips only; hard clips are not in
        the stored sequence)."""
        off = 0
        for op, l in self.cigartuples:
            if op == 4:
                off += l
            elif op == 5:
                continue
            else:
                break
        return off

    @property
    def query_alignment_end(self):
        end = self.query_length
        for op, l in reversed(self.cigartuples):
            if op == 4:
                end -= l
            elif op == 5:
                continue
            else:
                break
        return end


# -------------------------------------------------------------------------------------------------
# BGZF
# -------------------------------------------------------------------------------------------------
class BGZFReader:
    """Random access over BGZF blocks by virtual offset (coffset << 16 | uoffset)."""

    def __init__(self, path: str):
        self.path = path
        self.fh = open(path, "rb")
        self._block_coffset = -1
        self._block = b""
        self._next_coffset = 0
        self._pos = 0

    def close(self):
        self.fh.close()

    def _load_block(self, coffset: int) -> bool:
        self.fh.seek(coffset)
        head = self.fh.read(18)
        if len(head) < 18:
            self._block, self._block_coffset, self._next_coffset, self._pos = b"", coffset, coffset, 0
            if len(head):
                raise IOError("truncated BGZF block header at offset {}".format(coffset))
            return False
        id1, id2, cm, flg, _mtime, _xfl, _os, xlen = struct.unpack("<BBBBIBBH", head[:12])
        if id1 != 31 or id2 != 139 or not (flg & 4):
            raise ValueError("not a BGZF block at offset {}".format(coffset))
        extra = head[12:] + self.fh.read(xlen - 6)
        bsize = None
        off = 0
        while off + 4 <= len(extra):
            si1, si2, slen = struct.unpack_from("<BBH", extra, off)
            if si1 == 66 and si2 == 67:
                bsize = struct.unpack_from("<H", extra, off + 4)[0]
            off += 4 + slen
        if bsize is None:
            raise ValueError("BGZF block without BC subfield")
        cdata_len = bsize - xlen - 19
        cdata = self.fh.read(cdata_len)
        tail = self.fh.read(8)  # crc32 + isize
        if len(cdata) < cdata_len or len(tail) < 8:
            raise IOError("truncated BGZF block at offset {}".format(coffset))
        crc, isize = struct.unpack("<II", tail)
        self._block = zlib.decompress(cdata, -15) if cdata_len > 0 else b""
        # htslib / pysam verify both: a damaged block is an error, not data
        if len(self._block) != isize or (zlib.crc32(self._block) & 0xFFFFFFFF) != crc:
            raise IOError("corrupt BGZF block at offset {} (length / CRC-32)".format(coffset))
        self._block_coffset = coffset
        self._next_coffset = coffset + bsize + 1
        self._pos = 0
        return True

    def seek(self, voffset: int):
        coffset, uoffset = voffset >> 16, voffset & 0xFFFF
        if coffset != self._block_coffset:
            self._load_block(coffset)
        self._pos = uoffset

    def tell(self) -> int:
        if self._pos >= len(self._block) and self._block_coffset >= 0:
            return self._next_coffset << 16
        return (self._block_coffset << 16) | self._pos

    def read(self, n: int) -> bytes:
        out = []
        while n > 0:
            avail = len(self._block) - self._pos
            if avail <= 0:
                if not self._load_block(self._next_coffset):
                    break
                if not self._block:
                    if self._next_coffset == self._block_coffset:
                        break
                    continue
                avail = len(self._block)
            take = min(avail, n)
            out.append(self._block[self._pos:self._pos + take])
            self._pos += take
            n -= take
        return b"".join(out)


def bgzf_block(data: bytes, level: int = 6) -> bytes:
    """one BGZF block holding `data` (at most 0xFF00 bytes); blocks are independent, so they can be made in parallel"""
    comp = zlib.compressobj(level, zlib.DEFLATED, -15)
    cdata = comp.compress(data) + comp.flush()
    return (struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, len(cdata) + 25) + cdata +
            struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))


def bgzf_blocks(path: str) -> List[Tuple[int, int, int]]:
    """(compressed offset, inflated offset, inflated size) of every block of a BGZF file, from one walk of the block
    headers: BSIZE from each header, ISIZE from each block's last 4 bytes.  Nothing is inflated.  ValueError for a
    file that is not BGZF, IOError for a truncated one."""
    out = []
    coff = uoff = 0
    with open(path, "rb") as fh:
        size = os.fstat(fh.fileno()).st_size
        while coff < size:
            fh.seek(coff)
            head = fh.read(12)
            if len(head) < 12:
                raise IOError("{}: truncated BGZF block header at offset {}".format(path, coff))
            id1, id2, _cm, flg, _mtime, _xfl, _os, xlen = struct.unpack("<BBBBIBBH", head)
            if id1 != 31 or id2 != 139 or not (flg & 4):
                raise ValueError("{}: not a BGZF block at offset {}".format(path, coff))
            extra = fh.read(xlen)
            bsize, off = None, 0
            while off + 4 <= len(extra):
                si1, si2, slen = struct.unpack_from("<BBH", extra, off)
                if si1 == 66 and si2 == 67 and off + 6 <= len(extra):
                    bsize = struct.unpack_from("<H", extra, off + 4)[0] + 1
                off += 4 + slen
            if len(extra) < xlen:
                raise IOError("{}: truncated BGZF block header at offset {}".format(path, coff))
            if bsize is None or bsize < xlen + 20:
                raise ValueError("{}: BGZF block without a valid BC subfield at offset {}".format(path, coff))
            if coff + bsize > size:
                raise IOError("{}: truncated BGZF block at offset {}".format(path, coff))
            fh.seek(coff + bsize - 4)
            isize = struct.unpack("<I", fh.read(4))[0]
            out.append((coff, uoff, isize))
            coff += bsize
            uoff += isize
    return out


class BGZFWriter:
    """`block_size` uncompressed bytes per block (at most 0xFF00, what htslib uses, so a stored block fits)"""
    def __init__(self, path: str, level: int = 6, block_size: int = 0xFF00):
        if not 0 < block_size <= 0xFF00:
            raise ValueError("block_size must be in [1, 0xFF00]")
        self.fh = open(path, "wb")
        self.buf = bytearray()
        self.level = level
        self.block_size = block_size

    def write(self, data: bytes):
        self.buf += data
        n = self.block_size
        while len(self.buf) >= n:
            self._flush_block(bytes(self.buf[:n]))
            del self.buf[:n]

    def _flush_block(self, data: bytes):
        self.fh.write(bgzf_block(data, self.level))

    def tell(self) -> int:
        """Virtual offset of the next byte to be written."""
        return (self.fh.tell() << 16) | len(self.buf)

    def close(self):
        if self.buf:
            self._flush_block(bytes(self.buf))
            self.buf = bytearray()
        self._flush_block(b"")  # EOF marker
        self.fh.close()


# -------------------------------------------------------------------------------------------------
# BAI
# -------------------------------------------------------------------------------------------------
def _reg2bins(beg: int, end: int) -> List[int]:
    end -= 1
    bins = [0]
    for shift, offset in ((26, 1), (23, 9), (20, 73), (17, 585), (14, 4681)):
        bins.extend(range(offset + (beg >> shift), offset + (end >> shift) + 1))
    return bins


class BAIIndex:
    def __init__(self, path: str):
        data = open(path, "rb").read()
        if data[:4] != b"BAI\1":
            raise ValueError("not a BAI index: {}".format(path))
        off = 4
        (n_ref,) = struct.unpack_from("<i", data, off); off += 4
        self.bins = []
        self.linear = []
        for _ in range(n_ref):
            (n_bin,) = struct.unpack_from("<i", data, off); off += 4
            bins = {}
            for _ in range(n_bin):
                b, n_chunk = struct.unpack_from("<Ii", data, off); off += 8
                chunks = struct.unpack_from("<{}Q".format(2 * n_chunk), data, off); off += 16 * n_chunk
                bins[b] = [(chunks[2 * i], chunks[2 * i + 1]) for i in range(n_chunk)]
            (n_intv,) = struct.unpack_from("<i", data, off); off += 4
            ioff = struct.unpack_from("<{}Q".format(n_intv), data, off); off += 8 * n_intv
            self.bins.append(bins)
            self.linear.append(ioff)

    def chunks(self, tid: int, beg: int, end: int) -> List[Tuple[int, int]]:
        if tid >= len(self.bins):
            return []
        bins = self.bins[tid]
        lin = self.linear[tid]
        min_off = 0
        if lin:
            k = beg >> 14
            min_off = lin[k] if k < len(lin) else lin[-1]
        out = []
        for b in _reg2bins(beg, end):
            if b == 37450:  # metadata pseudo-bin
                continue
            for (s, e) in bins.get(b, ()):
                if e > min_off:
                    out.append((s, e))
        out.sort()
        merged = []
        for s, e in out:
            if merged and s <= merged[-1][1]:
                merged[-1] = (merged[-1][0], max(merged[-1][1], e))
            else:
                merged.append((s, e))
        return merged


# -------------------------------------------------------------------------------------------------
# BAM
# -------------------------------------------------------------------------------------------------
class AlignmentFile:
    """pysam.AlignmentFile stand-in (read mode)."""

    def __init__(self, path: str, mode: str = "rb"):
        if not os.path.exists(path):
            raise IOError("file `{}` not found".format(path))
        self.filename = path
        self.bgzf = BGZFReader(path)
        magic = self.bgzf.read(4)
        if magic != b"BAM\1":
            raise ValueError("not a BAM file: {}".format(path))
        (l_text,) = struct.unpack("<i", self.bgzf.read(4))
        self.text = self.bgzf.read(l_text).decode("latin-1")
        (n_ref,) = struct.unpack("<i", self.bgzf.read(4))
        self.references, self.lengths = [], []
        for _ in range(n_ref):
            (l_name,) = struct.unpack("<i", self.bgzf.read(4))
            name = self.bgzf.read(l_name)[:-1].decode("latin-1")
            (l_ref,) = struct.unpack("<i", self.bgzf.read(4))
            self.references.append(name)
            self.lengths.append(l_ref)
        self._tid = {n: i for i, n in enumerate(self.references)}
        self._first_record = self.bgzf.tell()
        self.index = None
        for cand in (path + ".bai", path.rsplit(".", 1)[0] + ".bai"):
            if os.path.exists(cand):
                self.index = BAIIndex(cand)
                break

    def close(self):
        self.bgzf.close()

    def getrname(self, tid: int) -> str:
        return self.references[tid]

    get_reference_name = getrname

    def get_tid(self, name: str) -> int:
        return self._tid.get(name, -1)

    # record decoding -----------------------------------------------------------------------------
    def _read_record(self) -> Optional[AlignedSegment]:
        head = self.bgzf.read(4)
        if len(head) < 4:
            return None
        (block_size,) = struct.unpack("<i", head)
        data = self.bgzf.read(block_size)
        if len(data) < block_size:
            return None
        (refID, pos, l_read_name, mapq, _bin, n_cigar, flag, l_seq, next_refID, next_pos,
         tlen) = struct.unpack_from("<iiBBHHHiiii", data, 0)
        off = 32
        name = data[off:off + l_read_name - 1].decode("latin-1"); off += l_read_name
        cig = struct.unpack_from("<{}I".format(n_cigar), data, off); off += 4 * n_cigar
        cigartuples = [(c & 0xF, c >> 4) for c in cig]
        nb = (l_seq + 1) // 2
        packed = np.frombuffer(data, dtype=np.uint8, count=nb, offset=off); off += nb
        seq = "".join(_NIB2[packed].tolist())[:l_seq] if l_seq else ""
        qual = data[off:off + l_seq]
        return AlignedSegment(name, flag, refID, pos, mapq, cigartuples, next_refID, next_pos, tlen,
                              seq, qual, aux=bytes(data[off + l_seq:]))

    # iteration -----------------------------------------------------------------------------------
    def fetch(self, contig: Optional[str] = None, start: Optional[int] = None,
              end: Optional[int] = None) -> Iterator[AlignedSegment]:
        """Records overlapping [start, end) (0-based, half-open) on ``contig`` in file order; all
        records when called without arguments.  Raises ValueError for an unknown contig, like pysam
        (``bam_parser.py:439-445`` relies on it)."""
        if contig is None:
            return self._iter_all()
        if contig not in self._tid:
            raise ValueError("invalid contig `{}`".format(contig))
        tid = self._tid[contig]
        if start is None:
            start = 0
        if end is None:
            end = self.lengths[tid]
        start = max(0, int(start))
        end = int(end)
        if self.index is not None:
            return self._iter_indexed(tid, start, end)
        return self._iter_scan(tid, start, end)

    def _iter_all(self):
        self.bgzf.seek(self._first_record)
        while True:
            r = self._read_record()
            if r is None:
                return
            yield r

    @staticmethod
    def _overlaps(r: AlignedSegment, start: int, end: int) -> bool:
        rend = r.reference_end
        if rend is None or rend <= r.reference_start:
            rend = r.reference_start + 1
        return r.reference_start < end and rend > start

    def _iter_scan(self, tid, start, end):
        # coordinate-sorted file: contigs ascend, unplaced (-1) records come last
        for r in self._iter_all():
            if r.reference_id != tid:
                if r.reference_id == -1 or r.reference_id > tid:
                    return
                continue
            if r.reference_start >= end:
                return
            if self._overlaps(r, start, end):
                yield r

    def _iter_indexed(self, tid, start, end):
        for (cbeg, cend) in self.index.chunks(tid, start, end):
            self.bgzf.seek(cbeg)
            while self.bgzf.tell() < cend:
                r = self._read_record()
                if r is None:
                    break
                if r.reference_id != tid:
                    if 0 <= r.reference_id < tid:
                        continue
                    return
                if r.reference_start >= end:
                    return
                if self._overlaps(r, start, end):
                    yield r


def region_depth(sam: AlignmentFile, chr: str, start: int, end: int) -> float:
    """Mean depth as ``BamDepth.region_depth`` computes it (``bam_parser.py:404-411``):
    ``sum(c.n for c in sam.pileup(chr, start, end)) / (end - start + 1)``.

    pysam's default pileup (``truncate=False``, ``stepper='all'``) walks every column covered by any
    read overlapping the window — including columns outside it — and skips UNMAP / SECONDARY /
    QCFAIL / DUP records; ``n`` counts reads spanning the column (deletions included).  The column
    sum therefore equals the total reference span of the qualifying overlapping reads.  pysam itself
    is not available to this build: these semantics are restated, not verified against pysam
    (SURVEY.md §8c, "depth is parity-unpinned")."""
    total = 0
    mask = FUNMAP | FSECONDARY | FQCFAIL | FDUP
    for r in sam.fetch(chr, start, end):
        if r.flag & mask:
            continue
        if not r.cigartuples:
            continue
        total += r.reference_length
    return total * 1.0 / (end - start + 1)


# -------------------------------------------------------------------------------------------------
# writer
# -------------------------------------------------------------------------------------------------
_ENC = {c: i for i, c in enumerate(_SEQ_DECODE)}


def _reg2bin(beg: int, end: int) -> int:
    end -= 1
    if beg >> 14 == end >> 14: return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17: return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20: return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23: return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26: return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def write_bam(path: str, references: List[Tuple[str, int]], records: List[AlignedSegment],
              header_text: Optional[str] = None, level: int = 6, index: bool = True, aux: bool = False):
    """Write a coordinate-sorted BAM (records must already be in file order) and, by default, its
    ``.bai`` index.  aux: write each record's raw optional fields (``AlignedSegment.aux``); without it records are
    written without any, as they always were."""
    w = BGZFWriter(path, level=level)
    bins = [dict() for _ in references]
    linear = [dict() for _ in references]
    if header_text is None:
        header_text = "@HD\tVN:1.4\tSO:coordinate\n" + "".join(
            "@SQ\tSN:{}\tLN:{}\n".format(n, l) for n, l in references)
    text = header_text.encode("latin-1")
    w.write(b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(references)))
    for name, length in references:
        nm = name.encode("latin-1") + b"\0"
        w.write(struct.pack("<i", len(nm)) + nm + struct.pack("<i", length))
    for r in records:
        nm = r.query_name.encode("latin-1") + b"\0"
        seq = r.query_sequence or ""
        l_seq = len(seq)
        codes = [_ENC.get(c.upper(), 15) for c in seq]
        if l_seq % 2:
            codes.append(0)
        packed = bytes((codes[i] << 4) | codes[i + 1] for i in range(0, len(codes), 2))
        qual = r._qual if (r._qual is not None and len(r._qual) == l_seq) else b"\xff" * l_seq
        cig = b"".join(struct.pack("<I", (l << 4) | op) for op, l in r.cigartuples)
        rend = r.reference_end
        if rend is None or rend <= r.reference_start:
            rend = r.reference_start + 1
        body = struct.pack("<iiBBHHHiiii", r.reference_id, r.reference_start, len(nm),
                           r.mapping_quality, _reg2bin(max(r.reference_start, 0), max(rend, 1)),
                           len(r.cigartuples), r.flag, l_seq, r.next_reference_id,
                           r.next_reference_start, r.template_length)
        body += nm + cig + packed + qual + ((r.aux or b"") if aux else b"")
        vbeg = w.tell()
        w.write(struct.pack("<i", len(body)) + body)
        vend = w.tell()
        if index and 0 <= r.reference_id < len(references):
            beg = max(r.reference_start, 0)
            b = _reg2bin(beg, max(rend, 1))
            chunks = bins[r.reference_id].setdefault(b, [])
            if chunks and chunks[-1][1] == vbeg:
                chunks[-1][1] = vend
            else:
                chunks.append([vbeg, vend])
            lin = linear[r.reference_id]
            for k in range(beg >> 14, ((max(rend, 1) - 1) >> 14) + 1):
                if k not in lin:
                    lin[k] = vbeg
    w.close()
    if index:
        with open(path + ".bai", "wb") as fh:
            fh.write(b"BAI\1" + struct.pack("<i", len(references)))
            for tid in range(len(references)):
                fh.write(struct.pack("<i", len(bins[tid])))
                for b in sorted(bins[tid]):
                    ch = bins[tid][b]
                    fh.write(struct.pack("<Ii", b, len(ch)))
                    for s_, e_ in ch:
                        fh.write(struct.pack("<QQ", s_, e_))
                lin = linear[tid]
                n_intv = (max(lin) + 1) if lin else 0
                fh.write(struct.pack("<i", n_intv))
                last = 0
                vals = []
                for k in range(n_intv):           # empty windows inherit the next filled offset
                    vals.append(lin.get(k, None))
                nxt = 0
                for k in range(n_intv - 1, -1, -1):
                    if vals[k] is None:
                        vals[k] = nxt
                    else:
                        nxt = vals[k]
                for v in vals:
                    fh.write(struct.pack("<Q", v))
