#!/usr/bin/env python
"""The scan of a BAM without an index (tredsw_ingest_scan_run) on a synthetic whole-sample BAM of at least 2 GB
inflated: background pairs tiled over every contig of the fixtures' reference dictionary, plus the reads of every
catalogue locus simulated by ``simulate.locus_records``.  Records are built with numpy and compressed on host threads
(zlib releases the GIL), so the file is written in about a minute; its .bai is built the same way.

Times, on the GPU the context runs on:
  * the scan of the unindexed copy: every catalogue locus with its alt regions and the chrY regions of the gender
    inference; total, host read and device time per slab, GB/s compressed and inflated, repaired blocks;
  * the indexed GPU ingest (tredsw_ingest_batch_run) of the same loci on the indexed file, whose evidence must equal
    the scan's problem by problem;
  * the Python reader (bam_parser.extract_locus) for HD without alt regions on the unindexed copy, once.
The card's name and power limit are printed with the numbers.  Everything is written to a temporary directory.

    python tools/scan_bench.py [--gb 2.2] [--slab-mb 0] [--reps 3] [--out result.json]
"""
import argparse
import json
import os
import shutil
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

READLEN, INSERT = 150, 350
NAME_LEN = 12                                  # "b" + 11 digits, NUL-terminated
REC_BYTES = 4 + 32 + (NAME_LEN + 1) + 4 + READLEN // 2 + READLEN
BLOCK = 0xFF00


def reg2bin(beg, end):
    """bamio._reg2bin on arrays (end exclusive)"""
    end = end - 1
    out = np.zeros(len(beg), np.int64)
    done = np.zeros(len(beg), bool)
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        hit = ~done & ((beg >> shift) == (end >> shift))
        out[hit] = off + (beg[hit] >> shift)
        done |= hit
    return out


def background(tid, length, n, rng, first_name):
    """n records of proper pairs tiled over one contig, sorted by position: (pos, raw record bytes)"""
    npairs = n // 2
    p1 = np.sort(rng.integers(0, max(1, length - INSERT - READLEN), npairs)).astype(np.int64)
    p2 = p1 + INSERT - READLEN
    pos = np.concatenate([p1, p2])
    mate = np.concatenate([p2, p1])
    flag = np.concatenate([np.full(npairs, 0x1 | 0x2 | 0x20 | 0x40), np.full(npairs, 0x1 | 0x2 | 0x10 | 0x80)])
    name = np.concatenate([np.arange(npairs), np.arange(npairs)]) + first_name
    tlen = np.concatenate([np.full(npairs, INSERT), np.full(npairs, -INSERT)])
    order = np.argsort(pos, kind="stable")
    pos, mate, flag, name, tlen = pos[order], mate[order], flag[order], name[order], tlen[order]
    m = len(pos)
    rec = np.zeros((m, REC_BYTES), np.uint8)
    head = np.zeros(m, np.dtype([("bs", "<i4"), ("tid", "<i4"), ("pos", "<i4"), ("ln", "u1"), ("mq", "u1"), ("bin", "<u2"),
                                 ("nc", "<u2"), ("flag", "<u2"), ("ls", "<i4"), ("nt", "<i4"), ("np", "<i4"), ("tl", "<i4")]))
    head["bs"] = REC_BYTES - 4; head["tid"] = tid; head["pos"] = pos; head["ln"] = NAME_LEN + 1; head["mq"] = 60
    head["bin"] = reg2bin(pos, pos + READLEN); head["nc"] = 1; head["flag"] = flag; head["ls"] = READLEN
    head["nt"] = tid; head["np"] = mate; head["tl"] = tlen
    rec[:, :36] = head.view(np.uint8).reshape(m, 36)
    digits = (name[:, None] // (10 ** np.arange(NAME_LEN - 2, -1, -1))) % 10
    rec[:, 36] = ord("b")
    rec[:, 37:36 + NAME_LEN] = (digits + ord("0")).astype(np.uint8)
    c = 36 + NAME_LEN + 1
    rec[:, c:c + 4] = np.frombuffer(struct.pack("<I", READLEN << 4), np.uint8)
    nib = np.array([1, 2, 4, 8], np.uint8)[rng.integers(0, 4, (m, READLEN))]
    rec[:, c + 4:c + 4 + READLEN // 2] = (nib[:, 0::2] << 4) | nib[:, 1::2]
    rec[:, c + 4 + READLEN // 2:] = np.array(list(b"IIIIHHGF#:"), np.uint8)[rng.integers(0, 10, (m, READLEN))]
    return pos, rec


def encode(r):
    """bamio.write_bam's record layout for one AlignedSegment"""
    from tredparse_b200 import bamio
    nm = r.query_name.encode("latin-1") + b"\0"
    seq = r.query_sequence
    codes = [bamio._ENC.get(ch, 15) for ch in seq] + ([0] if len(seq) % 2 else [])
    packed = bytes((codes[i] << 4) | codes[i + 1] for i in range(0, len(codes), 2))
    rend = r.reference_start + sum(l for op, l in r.cigartuples if op in (0, 2, 3, 7, 8))
    body = struct.pack("<iiBBHHHiiii", r.reference_id, r.reference_start, len(nm), r.mapping_quality,
                       int(reg2bin(np.array([r.reference_start]), np.array([rend]))[0]), len(r.cigartuples), r.flag,
                       len(seq), r.next_reference_id, r.next_reference_start, r.template_length)
    body += nm + b"".join(struct.pack("<I", (l << 4) | op) for op, l in r.cigartuples) + packed + b"\xff" * len(seq) + r.aux
    return struct.pack("<i", len(body)) + body, rend


def write_sample(path, gb, seed=5, extra=()):
    """-> (records, inflated bytes); writes path and path.bai.  extra: more bamio.AlignedSegment records (placed by
    contig and position; records without a contig go to the unmapped tail)"""
    from tredparse_b200 import bamio, simulate
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    sam = bamio.AlignmentFile(os.path.join(ROOT, "tests", "golden", "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    tid_of = {n: i for i, (n, _) in enumerate(refs)}
    rng = np.random.default_rng(seed)
    total_len = sum(l for _, l in refs)
    nrec = int(gb * 1e9 / REC_BYTES)
    text = ("@HD\tVN:1.4\tSO:coordinate\n" + "".join("@SQ\tSN:{}\tLN:{}\n".format(n, l) for n, l in refs)).encode()
    header = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for n, l in refs:
        header += struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", l)
    loci = {}
    for li, name in enumerate(repo.names):
        t = repo[name]
        if t.chr not in tid_of:
            continue
        sp = simulate.problem_spec(repo, repo.names, 0, li, READLEN, seed)
        for r in simulate.locus_records(t, tid_of[t.chr], tuple(sp["alleles"]), READLEN, sp["cov_per_hap"],
                                        seed=sp["seed"], tag="l{}".format(li)):
            raw, rend = encode(r)
            loci.setdefault(r.reference_id, []).append((r.reference_start, rend, raw))
    for r in extra:
        raw, rend = encode(r)
        loci.setdefault(r.reference_id, []).append((r.reference_start, rend, raw))
    # the stream, contig by contig: (per record) position, end, bytes in file order
    parts, meta = [header], []                     # meta: (tid, pos array, end array, lengths array)
    first_name = 0
    for tid, (name, length) in enumerate(refs):
        n = int(nrec * length / total_len) & ~1
        pos, rec = background(tid, length, n, rng, first_name)
        first_name += n
        lrecs = sorted(loci.get(tid, []), key=lambda x: x[0])
        lpos = np.array([x[0] for x in lrecs], np.int64)
        cut = np.searchsorted(pos, lpos, side="right")
        prev = 0
        P, E, L = [], [], []
        for k, (p, e, raw) in enumerate(lrecs):
            if cut[k] > prev:
                parts.append(rec[prev:cut[k]].tobytes())
                P.append(pos[prev:cut[k]]); E.append(pos[prev:cut[k]] + READLEN); L.append(np.full(cut[k] - prev, REC_BYTES))
                prev = cut[k]
            parts.append(raw)
            P.append(np.array([p])); E.append(np.array([max(e, p + 1)])); L.append(np.array([len(raw)]))
        if prev < len(pos):
            parts.append(rec[prev:].tobytes())
            P.append(pos[prev:]); E.append(pos[prev:] + READLEN); L.append(np.full(len(pos) - prev, REC_BYTES))
        meta.append((tid, np.concatenate(P) if P else np.zeros(0, np.int64), np.concatenate(E) if E else np.zeros(0, np.int64),
                     np.concatenate(L) if L else np.zeros(0, np.int64)))
    parts += [raw for _, _, raw in loci.get(-1, [])]          # the unmapped tail (not in the index)
    stream = b"".join(parts)
    del parts
    nblocks = (len(stream) + BLOCK - 1) // BLOCK

    def deflate(k):
        data = stream[k * BLOCK:(k + 1) * BLOCK]
        c = zlib.compressobj(1, zlib.DEFLATED, -15)
        cd = c.compress(data) + c.flush()
        return (struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, len(cd) + 25) + cd
                + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))
    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as pool:
        blocks = list(pool.map(deflate, range(nblocks)))
    coff = np.zeros(nblocks + 1, np.int64)
    coff[1:] = np.cumsum([len(b) for b in blocks])
    with open(path, "wb") as fh:
        for b in blocks:
            fh.write(b)
        fh.write(struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, 27) + b"\3\0" + b"\0" * 8)
    # the .bai, as bamio.write_bam builds it
    voff = lambda u: (coff[u // BLOCK] << 16) | (u % BLOCK)
    u = len(header)
    with open(path + ".bai", "wb") as fh:
        fh.write(b"BAI\1" + struct.pack("<i", len(refs)))
        for tid, pos, end, lens in meta:
            ustart = u + np.concatenate([[0], np.cumsum(lens)[:-1]]) if len(lens) else np.zeros(0, np.int64)
            u += int(lens.sum())
            vb, ve = voff(ustart), voff(ustart + lens)
            bins = reg2bin(pos, end)
            # chunks: runs of consecutive records of one bin, merged per bin in file order
            brk = np.flatnonzero(np.diff(bins)) + 1 if len(bins) else np.zeros(0, np.int64)
            r0 = np.concatenate([[0], brk]) if len(bins) else np.zeros(0, np.int64)
            r1 = np.concatenate([brk, [len(bins)]]) if len(bins) else np.zeros(0, np.int64)
            by_bin = {}
            for b, s_, e_ in zip(bins[r0].tolist(), vb[r0].tolist(), ve[r1 - 1].tolist()):
                ch = by_bin.setdefault(b, [])
                if ch and ch[-1][1] == s_:
                    ch[-1][1] = e_
                else:
                    ch.append([s_, e_])
            fh.write(struct.pack("<i", len(by_bin)))
            for b in sorted(by_bin):
                fh.write(struct.pack("<Ii", b, len(by_bin[b])))
                fh.write(np.array(by_bin[b], np.uint64).tobytes())
            if not len(pos):
                fh.write(struct.pack("<i", 0))
                continue
            nwin = int(((end - 1) >> 14).max()) + 1
            lin = np.full(nwin, np.iinfo(np.int64).max, np.int64)
            for k in range(int(((end - 1 - pos) >> 14).max()) + 1):        # windows a record covers
                w = (pos >> 14) + k
                ok = w <= ((end - 1) >> 14)
                np.minimum.at(lin, w[ok], vb[ok])
            empty = lin == np.iinfo(np.int64).max
            nxt = 0
            for k in range(nwin - 1, -1, -1):                              # empty windows inherit the next filled offset
                if empty[k]:
                    lin[k] = nxt
                else:
                    nxt = lin[k]
            fh.write(struct.pack("<i", nwin) + lin.astype("<u8").tobytes())
    return sum(len(m[1]) for m in meta) + len(loci.get(-1, [])), len(stream)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=2.2, help="inflated size of the synthetic BAM")
    ap.add_argument("--slab-mb", type=float, default=0, help="compressed MiB per slab (0: the library's default)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from tredparse_b200 import ingest, _lib, bam_parser
    from tredparse_b200.meta import TREDsRepo
    from tredparse_b200.bam_parser import BamDepth
    repo = TREDsRepo()
    res = {}
    try:
        res["card"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                     capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception as e:
        res["card"] = "unknown ({})".format(e)
    tmp = tempfile.mkdtemp(prefix="scan_bench_")
    try:
        path = os.path.join(tmp, "sample.bam")
        t = time.perf_counter()
        nrec, inflated = write_sample(path, a.gb)
        res.update(write_s=time.perf_counter() - t, records=nrec, inflated_bytes=inflated, file_bytes=os.path.getsize(path))
        unidx = os.path.join(tmp, "unindexed.bam")
        os.link(path, unidx)
        ctx = _lib.default_context(0)
        ih, uh = ingest.BamIngest(path), ingest.BamIngest.unindexed(unidx)
        names = list(repo.names)
        qs, keep = [], []
        for n in names:
            q = ingest.locus_query(uh, repo[n], READLEN, alts=repo[n].alt)
            qs.append(q[0]); keep.append(q[1])
        yreg = [(uh.tid(c), s, e) for c, s, e in BamDepth.y_regions(repo.ref)]
        slab = int(a.slab_mb * (1 << 20)) or None
        scans = []
        for _ in range(a.reps):
            t = time.perf_counter()
            b = ingest.scan_sample(ctx, uh, qs, keep, yreg, slab_bytes=slab)
            wall = time.perf_counter() - t
            st = b.stats()
            st["wall_s"] = wall
            scans.append(st)
            if _ < a.reps - 1:
                b.close()
        best = min(scans, key=lambda s: s["wall_s"])
        res["scan"] = {"runs": scans, "best_wall_s": best["wall_s"],
                       "GBps_compressed": best["compressed_bytes"] / best["wall_s"] / 1e9,
                       "GBps_inflated": best["inflated_bytes"] / best["wall_s"] / 1e9,
                       "ms_host_read_per_slab": best["ms_host_read"] / best["slabs"],
                       "ms_device_per_slab": best["ms_device"] / best["slabs"],
                       "bound_by": "device" if best["ms_device"] > best["ms_host_read"] else "host read",
                       "status": int(b.scan_status), "problems_flagged": int((b.status != 0).sum()),
                       "depthY": float(np.median(b.depths))}
        # the indexed GPU ingest of the same loci; equal evidence problem by problem
        times = []
        for _ in range(a.reps):
            t = time.perf_counter()
            ib = ingest.IngestBatch(ctx, [ih], [0] * len(qs), qs, keep=keep)
            times.append(time.perf_counter() - t)
            if _ < a.reps - 1:
                ib.close()
        bad = 0
        for i in range(len(qs)):
            x, y = b.evidence(i), ib.evidence(i)
            bad += not (np.array_equal(x.reads, y.reads) and np.array_equal(x.roff, y.roff) and x.names == y.names
                        and np.array_equal(x.global_lens, y.global_lens) and np.array_equal(x.target_lens, y.target_lens)
                        and x.depth == y.depth and x.n_unmapped == y.n_unmapped)
        assert not ib.status.any() and not b.status.any() and bad == 0, "the scan and the indexed ingest differ"
        res["indexed_ingest"] = {"best_s": min(times), "runs_s": times, "stats": ib.stats(), "reads": int(ib.nreads)}
        res["problems"], res["problems_differing"] = len(qs), bad
        ib.close(); b.close()
        # the Python reader, one locus without alt regions, once
        import logging
        t = time.perf_counter()
        ev = bam_parser.extract_locus(unidx, repo, "HD", READLEN, False, False, logging.getLogger())
        res["python_reader_HD_no_alts_s"] = time.perf_counter() - t
        res["python_reader_HD_reads"] = ev.nreads
        ih.close(); uh.close()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fp:
            fp.write(line + "\n")


if __name__ == "__main__":
    main()
