"""GPU BAM ingest (csrc/bgzf_gpu.cu, csrc/ingest_device.cuh): BGZF inflate, record walk, read selection, pairing
by name and depth for a whole batch of (sample, locus) problems — against the host reader
(tredsw_bam_extract_locus, itself pinned to the Python reader and the reference's BAMs in test_ingest.py).

CPU tests run the SAME per-thread bodies through the serial host backend (tredsw_ingest_batch_emulate: test
infrastructure); the `gpu` tests run the kernels and compare with the host reader problem by problem."""
import os
import random
import shutil
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def repo():
    from tredparse_b200.meta import TREDsRepo
    return TREDsRepo()


def _queries(handles, repo, names, readlen=150, alts=True):
    from tredparse_b200 import ingest
    qs, so, keep, key = [], [], [], []
    for si, h in enumerate(handles):
        for n in names:
            q = ingest.locus_query(h, repo[n], readlen, alts=repo[n].alt if alts else ())
            if q is None:
                continue
            qs.append(q[0]); keep.append(q[1]); so.append(si); key.append((si, n))
    return qs, so, keep, key


def _same(ev, ref):
    return (np.array_equal(ev.reads, ref.reads) and np.array_equal(ev.roff, ref.roff)
            and np.array_equal(ev.global_lens, ref.global_lens) and np.array_equal(ev.target_lens, ref.target_lens)
            and ev.depth == ref.depth and ev.n_unmapped == ref.n_unmapped and ev.names == ref.names)


def _check_batch(ctx, paths, repo, names, alts=True, readlen=150):
    from tredparse_b200 import ingest
    hs = [ingest.BamIngest(p) for p in paths]
    try:
        qs, so, keep, key = _queries(hs, repo, names, readlen, alts)
        with ingest.IngestBatch(ctx, hs, so, qs, keep=keep) as b:
            assert b.nproblems == len(key) and not b.status.any()
            total = 0
            for i, (si, n) in enumerate(key):
                ref = hs[si].extract_locus(repo[n], readlen, alts=repo[n].alt if alts else (), want_names=True)
                assert _same(b.evidence(i), ref), (paths[si], n)
                total += ref.nreads
            st = b.stats()
            assert st["blocks"] > 0 and st["records"] > 0
            return total
    finally:
        for h in hs:
            h.close()


def _write_sample(path, repo, names, sample, seed, readlen=150):
    from tredparse_b200 import simulate, bamio
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    simulate.write_sample_bam(path, repo, names, refs, sample, readlen, seed)


def _raw_deflate(data, level, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    return c.compress(data) + c.flush()


# ---- CPU: the device code, executed serially on the host -----------------------------------------------------
def test_device_decoder_on_every_block_type():
    """stored / fixed / dynamic blocks, long distances, runs, every window size, empty input, and refusal of
    truncated or corrupted streams (the __host__ __device__ decoder behind inflate_kernel)."""
    from tredparse_b200 import _lib, ingest
    lib = _lib.load()
    ingest._bind_batch(lib)
    rng = random.Random(5)
    cases = [b"", b"a", b"ab" * 40000, bytes(rng.getrandbits(8) for _ in range(20000)),
             b"".join(bytes([rng.choice(b"ACGT")]) for _ in range(65536)),
             bytes(rng.choice(b"IIIIIHHGF#") for _ in range(30000)), open(__file__, "rb").read(), bytes(65536)]
    for data in cases:
        for level, strategy in ((0, 0), (1, 0), (6, 0), (9, 0), (6, zlib.Z_FIXED), (6, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE)):
            raw = _raw_deflate(data, level, strategy)
            out = np.zeros(len(data) + 16, np.uint8)
            assert lib.tredsw_inflate_raw_device_code(raw, len(raw), out.ctypes.data, len(data)) == 0
            assert bytes(out[:len(data)]) == data
            if len(data) > 100:
                # wrong inflated size, truncation, and bit flips must be refused or yield different bytes — never crash
                assert lib.tredsw_inflate_raw_device_code(raw, len(raw), out.ctypes.data, len(data) - 1) != 0
                assert lib.tredsw_inflate_raw_device_code(raw[:len(raw) // 2], len(raw) // 2, out.ctypes.data, len(data)) != 0
                for _ in range(20):
                    bad = bytearray(raw)
                    bad[rng.randrange(len(bad))] ^= 1 << rng.randrange(8)
                    rc = lib.tredsw_inflate_raw_device_code(bytes(bad), len(bad), out.ctypes.data, len(data))
                    assert rc != 0 or zlib.crc32(bytes(out[:len(data)])) != zlib.crc32(data) or bytes(out[:len(data)]) == data


def test_emulated_pipeline_equals_host_reader_on_the_fixtures(repo):
    paths = [os.path.join(GOLDEN, "t001.mini.bam"), os.path.join(GOLDEN, "t002.mini.bam")]
    assert _check_batch(None, paths, repo, repo.names) > 100
    assert _check_batch(None, paths[:1], repo, ["HD"], alts=False) > 50
    assert _check_batch(None, paths, repo, ["HD", "DM1", "SCA17"], readlen=101) > 50


def test_emulated_pipeline_on_a_synthetic_whole_sample_bam(repo, tmp_path):
    """~30x at every catalogue locus: thousands of pair candidates per problem (pairing tables, ordered compaction);
    150 and 251 bp reads (the read window and the selection rules depend on the read length)."""
    names = ["HD", "DM1", "FXS", "SCA10"]
    for readlen in (150, 251):
        path = str(tmp_path / "s{}.bam".format(readlen))
        _write_sample(path, repo, names, 3, 11, readlen)
        assert _check_batch(None, [path], repo, names, readlen=readlen) > 200


def test_corrupt_input_is_reported_per_problem_not_as_evidence(repo, tmp_path):
    """a flipped byte inside a BGZF block / a truncated file: status != 0 for the problems of that sample, the other
    sample of the batch is untouched (the caller reads flagged problems with the host reader)."""
    from tredparse_b200 import ingest
    good = os.path.join(GOLDEN, "t001.mini.bam")
    for how in ("flip", "truncate"):
        bad = str(tmp_path / (how + ".bam"))
        data = bytearray(open(good, "rb").read())
        if how == "flip":
            data[len(data) // 2] ^= 0x55
        else:
            data = data[:len(data) // 2]
        open(bad, "wb").write(bytes(data))
        shutil.copy(good + ".bai", bad + ".bai")
        hs = [ingest.BamIngest(good), ingest.BamIngest(bad)]
        qs, so, keep, key = _queries(hs, repo, ["HD"])
        with ingest.IngestBatch(None, hs, so, qs, keep=keep) as b:
            assert b.status[0] == 0 and b.status[1] != 0
            assert _same(b.evidence(0), hs[0].extract_locus(repo["HD"], 150, alts=repo["HD"].alt, want_names=True))
        for h in hs:
            h.close()


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_ingest_equals_host_reader_on_the_fixtures(repo):
    from tredparse_b200 import _lib
    ctx = _lib.default_context(0)
    paths = [os.path.join(GOLDEN, "t001.mini.bam"), os.path.join(GOLDEN, "t002.mini.bam")]
    assert _check_batch(ctx, paths, repo, repo.names) > 100
    assert _check_batch(ctx, paths, repo, ["HD", "DM1"], alts=False) > 50


@pytest.mark.gpu
def test_gpu_ingest_on_synthetic_whole_sample_bams(repo, tmp_path):
    from tredparse_b200 import _lib
    ctx = _lib.default_context(0)
    names = [n for n in repo.names][:12]
    paths = []
    for s in range(3):
        p = str(tmp_path / "s{}.bam".format(s))
        _write_sample(p, repo, names, s, 21)
        paths.append(p)
    assert _check_batch(ctx, paths, repo, names) > 1000


@pytest.mark.gpu
def test_gpu_ingest_flags_corrupt_blocks(repo, tmp_path):
    from tredparse_b200 import _lib, ingest
    ctx = _lib.default_context(0)
    good = os.path.join(GOLDEN, "t001.mini.bam")
    bad = str(tmp_path / "flip.bam")
    data = bytearray(open(good, "rb").read())
    data[len(data) // 2] ^= 0x55
    open(bad, "wb").write(bytes(data))
    shutil.copy(good + ".bai", bad + ".bai")
    hs = [ingest.BamIngest(good), ingest.BamIngest(bad)]
    qs, so, keep, key = _queries(hs, repo, ["HD"])
    with ingest.IngestBatch(ctx, hs, so, qs, keep=keep) as b:
        assert b.status[0] == 0 and b.status[1] != 0
        assert _same(b.evidence(0), hs[0].extract_locus(repo["HD"], 150, alts=repo["HD"].alt, want_names=True))
    for h in hs:
        h.close()


@pytest.mark.gpu
def test_run_chunk_is_served_by_the_gpu_ingest_and_equals_the_host_reader_path(repo, tmp_path, monkeypatch):
    """tred.run_chunk on whole-sample BAMs: every locus comes from the GPU ingest (the host reader is not called),
    and the JSON fields equal those of the same run with the host reader (TREDSW_GPU_INGEST=0 behaviour)."""
    from tredparse_b200 import tred as T
    names = [n for n in repo.names][:10]
    paths = []
    for s in range(2):
        p = str(tmp_path / "s{}.bam".format(s))
        _write_sample(p, repo, names, s, 31)
        paths.append(p)
    tasks = [("s{}".format(i), p, repo, list(names), 300, False, False, True, True, "INFO") for i, p in enumerate(paths)]
    monkeypatch.setattr(T, "GPU_INGEST", False)
    host = T.run_chunk(tasks)
    monkeypatch.setattr(T, "GPU_INGEST", True)

    def no_host_reader(*a, **k):
        raise AssertionError("the host reader was called although the GPU ingest can serve every locus")
    monkeypatch.setattr(T, "ingest_loci", no_host_reader)
    # ... and the fused call runs on the ingest's device buffers (no batch assembled on the host, no second upload)
    from tredparse_b200 import cohort
    used = {"ingest": 0, "host": 0}
    run_host = cohort.CohortBatch.run_host

    def counted_host(self, *a, **k):
        used["ingest" if k.get("device_view") is not None else "host"] += 1
        return run_host(self, *a, **k)
    monkeypatch.setattr(cohort.CohortBatch, "run_host", counted_host)
    gpu = T.run_chunk(tasks)
    assert used == {"ingest": 1, "host": 0}
    for flags in ((True, True, False), (False, True, True)):          # --useclippedreads; --norepeatpairs (name ids)
        t2 = [x[:6] + flags + x[9:] for x in tasks]
        monkeypatch.setattr(T, "DEVICE_HANDOFF", False)
        a = T.run_chunk(t2)
        monkeypatch.setattr(T, "DEVICE_HANDOFF", True)
        b = T.run_chunk(t2)
        assert [r["tredCalls"] for r in a] == [r["tredCalls"] for r in b]
    assert used == {"ingest": 3, "host": 2}
    assert len(gpu) == len(host) == 2
    for a, b in zip(gpu, host):
        assert a["tredCalls"].keys() == b["tredCalls"].keys() and len(a["tredCalls"]) > 20 * len(names)
        assert a["tredCalls"] == b["tredCalls"]


def test_device_decoder_differential_fuzz_against_zlib():
    """randomised streams with shallow, deep (Fibonacci-weighted: 15-bit codes, sub-tables) and degenerate Huffman
    trees, every zlib strategy / level / memLevel: the device decoder returns zlib's input, byte for byte"""
    from tredparse_b200 import _lib, ingest
    lib = _lib.load()
    ingest._bind_batch(lib)
    rng = random.Random(123)
    nrng = np.random.default_rng(5)

    def gen(kind, n):
        if kind == 0:
            return bytes(nrng.integers(0, 256, n, dtype=np.uint8))
        if kind == 1:
            return bytes(np.minimum(nrng.geometric(rng.choice([0.3, 0.5, 0.7, 0.9]), n) - 1, 255).astype(np.uint8))
        if kind == 2:
            return bytes(np.minimum(nrng.zipf(rng.choice([1.2, 1.5, 2.0]), n), 255).astype(np.uint8))
        if kind == 3:
            unit = bytes(nrng.integers(0, 4, rng.randint(1, 300), dtype=np.uint8))
            b = bytearray(unit * (n // len(unit) + 1))[:n]
            for _ in range(n // 50):
                b[rng.randrange(n)] = rng.randrange(256)
            return bytes(b)
        if kind == 4:
            f, syms = [1, 1], []
            while len(f) < 24:
                f.append(f[-1] + f[-2])
            for i, c in enumerate(f):
                syms += [i] * min(c, 4000)
            rng.shuffle(syms)
            return bytes(syms[:n])
        return b"ACGT"[rng.randrange(4):][:1] * n
    for _ in range(400):
        data = gen(rng.randrange(6), rng.choice([1, 2, 10, 100, 1000, 5000, 20000, 65536]))
        c = zlib.compressobj(rng.choice([1, 4, 6, 9]), zlib.DEFLATED, -15, rng.choice([1, 5, 8, 9]),
                             rng.choice([zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]))
        raw = c.compress(data) + c.flush()
        out = np.zeros(len(data) + 16, np.uint8)
        assert lib.tredsw_inflate_raw_device_code(raw, len(raw), out.ctypes.data, len(data)) == 0
        assert bytes(out[:len(data)]) == data


def test_problem_records_built_from_an_ingest_batch_equal_the_host_assembled_batch(repo):
    """cohort.CohortBatch.from_ingest (the device hand-off: no concatenation, only the 40-byte problem records) against
    the batch assembled from the per-problem evidence — records, sizes, family tables, name ids (emulated ingest)"""
    from tredparse_b200 import ingest, cohort
    from tredparse_b200.simulate import Problem
    paths = [os.path.join(GOLDEN, "t001.mini.bam"), os.path.join(GOLDEN, "t002.mini.bam")]
    hs = [ingest.BamIngest(p) for p in paths]
    names = ["HD", "DM1", "SCA17", "AR"]
    qs, so, keep, key = _queries(hs, repo, names)
    with ingest.IngestBatch(None, hs, so, qs, keep=keep) as b:
        evs = [b.evidence(i) for i in range(len(key))]
        problems, fam_keys, fam_of = [], [], []
        for (si, n), ev in zip(key, evs):
            pr = Problem()
            pr.tred, pr.readlen, pr.ploidy, pr.depth = repo[n], 150, repo[n].ploidy, ev.depth
            pr.reads, pr.roff, pr.global_lens, pr.target_lens, pr.alleles, pr.names = ev.reads, ev.roff, ev.global_lens, ev.target_lens, None, ev.names
            problems.append(pr)
            if (repo[n], 150) not in fam_keys:
                fam_keys.append((repo[n], 150))
            fam_of.append(fam_keys.index((repo[n], 150)))
        for kw in ({}, {"repeatpairs": False}):
            host = cohort.CohortBatch(problems, **kw)
            dev = cohort.CohortBatch.from_ingest(b, np.array(fam_of, np.int32), np.array([p.ploidy for p in problems], np.int32),
                                                 np.array([p.depth for p in problems]), fam_keys,
                                                 names=[ev.names for ev in evs], **kw)
            assert dev.problems.tobytes() == host.problems.tobytes()
            assert (dev.nproblems, dev.nreads, dev.max_read_len) == (host.nproblems, host.nreads, host.max_read_len)
            assert len(dev.rbuf) == len(host.rbuf) and len(dev.pe_lens) == len(host.pe_lens)
            assert np.array_equal(dev.rbuf, host.rbuf) and np.array_equal(dev.roff, host.roff) and np.array_equal(dev.pe_lens, host.pe_lens)
            assert dev.families.tobytes() == host.families.tobytes() and dev.loci.tobytes() == host.loci.tobytes()
            assert (dev.read_name is None) == (host.read_name is None)
            if host.read_name is not None:
                assert np.array_equal(dev.read_name, host.read_name)
    for h in hs:
        h.close()


def _bam_with_a_corrupt_record(dst):
    """t001.mini.bam with ONE record whose l_seq does not fit its block_size, inside a BGZF block that is otherwise
    valid: the block is re-deflated, its CRC-32 recomputed, and a padding subfield keeps its size (and thus every
    virtual offset of the .bai) unchanged — corruption that only record-level checks can see."""
    import bisect
    import struct
    src = os.path.join(GOLDEN, "t001.mini.bam")
    data = open(src, "rb").read()
    blocks, o = [], 0
    while o < len(data):
        xlen = struct.unpack_from("<H", data, o + 10)[0]
        bsize = struct.unpack_from("<H", data, o + 16)[0] + 1
        blocks.append((o, xlen, bsize))
        o += bsize
    inflated, offs = b"", []
    for (o, xlen, bsize) in blocks:
        offs.append(len(inflated))
        inflated += zlib.decompress(data[o + 12 + xlen:o + bsize - 8], -15)
    p = 4
    p += 4 + struct.unpack_from("<i", inflated, p)[0]
    n_ref = struct.unpack_from("<i", inflated, p)[0]
    p += 4
    for _ in range(n_ref):
        p += 4 + struct.unpack_from("<i", inflated, p)[0] + 4
    recs = []
    while p + 4 <= len(inflated):
        recs.append(p)
        p += 4 + struct.unpack_from("<i", inflated, p)[0]
    for ri in range(len(recs) // 2, len(recs)):
        bi = bisect.bisect_right(offs, recs[ri]) - 1
        o, xlen, bsize = blocks[bi]
        raw = bytearray(inflated[offs[bi]:offs[bi + 1] if bi + 1 < len(offs) else len(inflated)])
        local = recs[ri] - offs[bi]
        if local + 300 > len(raw):
            continue
        struct.pack_into("<i", raw, local + 4 + 16, 0x7fffff00)                    # l_seq far beyond block_size
        for k in range(local + 120, local + 260):
            raw[k] = raw[local + 120]                                              # (more compressible: room for padding)
        for lvl, ml in ((9, 8), (9, 9), (8, 8)):
            c = zlib.compressobj(lvl, zlib.DEFLATED, -15, ml)
            cd = c.compress(bytes(raw)) + c.flush()
            pad = (bsize - 12 - xlen - 8) - len(cd)
            if pad == 0 or pad >= 4:
                extra = data[o + 12:o + 12 + xlen] + (b"ZZ" + struct.pack("<H", pad - 4) + b"\0" * (pad - 4) if pad else b"")
                hdr = bytearray(data[o:o + 12])
                struct.pack_into("<H", hdr, 10, len(extra))
                blk = bytes(hdr) + extra + cd + struct.pack("<II", zlib.crc32(bytes(raw)) & 0xffffffff, len(raw))
                assert len(blk) == bsize
                open(dst, "wb").write(data[:o] + blk + data[o + bsize:])
                shutil.copy(src + ".bai", dst + ".bai")
                return
    raise AssertionError("could not craft the file")


def _corrupt_record_case(ctx, repo, tmp_path):
    from tredparse_b200 import ingest, _lib
    bad = str(tmp_path / "corrupt_record.bam")
    _bam_with_a_corrupt_record(bad)
    good = os.path.join(GOLDEN, "t001.mini.bam")
    hs = [ingest.BamIngest(good), ingest.BamIngest(bad)]
    with pytest.raises(_lib.TredswError, match="corrupt BAM record"):          # the host reader refuses the file ...
        hs[1].extract_locus(repo["HD"], 150, alts=repo["HD"].alt, want_names=True)
    qs, so, keep, key = _queries(hs, repo, ["HD"])
    with ingest.IngestBatch(ctx, hs, so, qs, keep=keep) as b:                  # ... and the device code flags the problem
        assert b.status[0] == 0 and b.status[1] == 3
        assert _same(b.evidence(0), hs[0].extract_locus(repo["HD"], 150, alts=repo["HD"].alt, want_names=True))
    for h in hs:
        h.close()


def test_a_corrupt_record_inside_a_valid_block_is_flagged_emulated(repo, tmp_path):
    _corrupt_record_case(None, repo, tmp_path)


@pytest.mark.gpu
def test_a_corrupt_record_inside_a_valid_block_is_flagged_on_the_gpu(repo, tmp_path):
    from tredparse_b200 import _lib
    _corrupt_record_case(_lib.default_context(0), repo, tmp_path)


_STAGE_FUZZ = r"""
import os, sys, random, shutil
sys.path.insert(0, {root!r})
import numpy as np
from tredparse_b200 import ingest, _lib
from tredparse_b200.meta import TREDsRepo
repo = TREDsRepo()
good = open({bam!r}, "rb").read()
bai = open({bam!r} + ".bai", "rb").read()
rng = random.Random(11)
ok = flagged = refused = 0
for trial in range(120):
    bad, ix = bytearray(good), bytearray(bai)
    how = trial % 4
    if how == 0:                                           # bytes anywhere in the file: headers, payloads, footers
        for _ in range(rng.randrange(1, 6)):
            p = rng.randrange(len(bad)); bad[p] = rng.randrange(256)
    elif how == 1:                                         # truncated file
        bad = bad[:rng.randrange(100, len(bad))]
    elif how == 2:                                         # damaged index: chunk offsets point anywhere
        for _ in range(rng.randrange(1, 6)):
            p = rng.randrange(8, len(ix)); ix[p] = rng.randrange(256)
    else:                                                  # BGZF framing fields (XLEN, BSIZE, ISIZE) of some block
        off = 0
        for _ in range(rng.randrange(0, 25)):
            nxt = off + int.from_bytes(bad[off + 16:off + 18], "little") + 1
            if nxt + 28 >= len(bad): break
            off = nxt
        p = off + rng.choice([10, 11, 16, 17]); bad[p] = rng.randrange(256)
    p2 = os.path.join({tmp!r}, "bad.bam")
    open(p2, "wb").write(bytes(bad)); open(p2 + ".bai", "wb").write(bytes(ix))
    try:
        h = ingest.BamIngest(p2)
    except Exception:
        refused += 1
        continue
    try:
        qs = [ingest.locus_query(h, repo[n], 150, alts=repo[n].alt) for n in ("HD", "SCA17")]
        qs = [q for q in qs if q is not None]
        with ingest.IngestBatch(None, [h], [0] * len(qs), [q[0] for q in qs], keep=[q[1] for q in qs]) as b:
            for i in range(len(qs)):
                if b.status[i]:
                    flagged += 1
                else:
                    ev = b.evidence(i); assert ev.nreads == len(ev.roff) - 1 and ev.roff[-1] == len(ev.reads)
                    ok += 1
    except _lib.TredswError:
        refused += 1
    finally:
        h.close()
print("survived", ok, flagged, refused)
"""


def test_damaged_files_and_indexes_do_not_take_the_ingest_down(tmp_path):
    """the host staging (BAI chunks -> block ranges -> BGZF framing) and the device code (emulated) on damaged BAMs and
    damaged .bai files: every outcome is a result, a per-problem flag or a TredswError — never a crash"""
    import subprocess
    import sys
    code = _STAGE_FUZZ.format(root=ROOT, bam=os.path.join(GOLDEN, "t001.mini.bam"), tmp=str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-500:], r.stderr[-2000:])
    assert "survived" in r.stdout
