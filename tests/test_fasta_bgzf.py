"""Discovered loci from a bgzipped reference (DESIGN §4.5.1): `Fasta` on a BGZF file against the same text as plain
FASTA (index with and without .fai, lengths, fetch), the tract scan with its blocks inflated (host emulation; on the
GPU the kernels) against the plain-text scan and oracle/tract_oracle.py, the exact step plan over shared blocks,
corrupt, truncated and mis-indexed files, and `strprofile loci [--alts]` on a bgzipped reference."""
import gzip
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from test_ref_tracts import MOTIFS, _as_tuples, _big_fasta, _random_contigs, _write

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENV = dict(os.environ, PYTHONPATH=ROOT)

WIDTHS = [(1, False), (60, False), (61, False), (80, False), (60, True)]
BLOCKS = [97, 1000, 0xFF00]
LEVELS = [0, 1, 9]                  # stored DEFLATE blocks; dynamic-Huffman ones, and fixed ones in 97-byte blocks
STATS = ("steps", "bases", "invalid_bases", "tracts")

_oracle_cache = {}


def _contigs(width, crlf):
    return _random_contigs(width + 1000 * crlf)


def _oracle(width, crlf):
    from oracle import tract_oracle
    if (width, crlf) not in _oracle_cache:
        _oracle_cache[(width, crlf)] = tract_oracle.tracts(_contigs(width, crlf), MOTIFS, 3, 30)
    return _oracle_cache[(width, crlf)]


def _pair(tmp_path, contigs, width, crlf=False, block=0xFF00, level=6, fai=False):
    """(plain Fasta, BGZF Fasta) of one text"""
    from tredparse_b200 import simulate
    from tredparse_b200.fasta import Fasta
    plain = _write(str(tmp_path / "r.fa"), contigs, width, crlf)
    if fai:
        idx = Fasta(plain).index
        with open(plain + ".fai", "w") as fp:
            fp.writelines("{}\t{}\t{}\t{}\t{}\n".format(n, *e) for n, e in idx.items())
    gz = simulate.bgzip_fasta(plain, str(tmp_path / "r.fa.gz"), block_size=block, level=level)
    assert os.path.exists(gz + ".fai") == fai
    return Fasta(plain), Fasta(gz)


def _plan(fa, step_bytes):
    """the step plan of a scan: contigs under the text budget (as tredsw_ref_tracts groups them), then per step the
    blocks from the one holding its first text byte to the one holding its last -> (steps, inflated bytes,
    compressed bytes, blocks)"""
    import bisect
    budget = step_bytes or 256 << 20
    groups = []
    for e in fa.index.values():
        L, off, lb, lw = e
        n = (L - 1) // lb * lw + (L - 1) % lb + 1 if L > 0 else 0
        if not groups or (groups[-1][0] + n > budget and groups[-1][1]):
            groups.append([0, []])
        groups[-1][0] += n
        groups[-1][1].append((off, n))
    starts = [b[1] for b in fa.blocks]
    coffs = [b[0] for b in fa.blocks] + [os.path.getsize(fa.path)]
    inflated = comp = blocks = 0
    for _, cs in groups:
        cs = [(off, n) for off, n in cs if n]
        if not cs:
            continue
        b0 = bisect.bisect_right(starts, min(off for off, _ in cs)) - 1
        b1 = bisect.bisect_right(starts, max(off + n - 1 for off, n in cs))
        inflated += fa.blocks[b1 - 1][1] + fa.blocks[b1 - 1][2] - fa.blocks[b0][1]
        comp += coffs[b1] - coffs[b0]
        blocks += b1 - b0
    return len(groups), inflated, comp, blocks


def _check_plan(res, fa, step_bytes):
    st = res["stats"]
    assert (st["steps"], st["bytes"], st["comp_bytes"], st["blocks"]) == _plan(fa, step_bytes)


# ---------------------------------------------------------------------------------------------------------------
# Fasta: index, lengths and fetch on a BGZF file == on the plain text
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width,crlf", WIDTHS)
@pytest.mark.parametrize("block", BLOCKS)
def test_fasta_on_bgzf_equals_the_plain_text(tmp_path, width, crlf, block):
    from tredparse_b200.fasta import Fasta
    contigs = _contigs(width, crlf)
    contigs["inside"] = "ACGTACGTNNacgt"               # a contig that begins and ends inside one block
    for level in LEVELS:
        for fai in (False, True):
            d = tmp_path / "l{}f{}".format(level, int(fai))
            d.mkdir()
            plain, gz = _pair(d, contigs, width, crlf, block, level, fai)
            assert gz.blocks is not None and plain.blocks is None and len(gz.blocks) > (1 if block < 0xFF00 else 0)
            assert gz.index == plain.index == Fasta(plain.path).index
            assert gz.lengths() == plain.lengths() == {n: len(s) for n, s in contigs.items()}
            rng = np.random.default_rng(block + level + width)
            for n, s in contigs.items():
                assert gz.fetch(n, 0, len(s)) == s.upper()
                assert gz.fetch(n, -5, 3) == s[:3].upper() and gz.fetch(n, len(s) - 2, len(s) + 9) == s[-2:].upper()
                for _ in range(20):
                    a = int(rng.integers(0, len(s) + 1))
                    b = int(rng.integers(a, len(s) + 1))
                    assert gz.fetch(n, a, b) == plain.fetch(n, a, b) == s[a:b].upper()
            if block == 97:                            # windows that straddle every block boundary of one contig
                L, off, lb, lw = gz.index["ctg1"]
                for _, u, _ in gz.blocks:
                    if off < u < off + L:
                        i = (u - off) // lw * lb + min((u - off) % lw, lb)     # the base at or after the boundary
                        assert gz.fetch("ctg1", i - 3, i + 3) == contigs["ctg1"][max(0, i - 3):i + 3].upper()
            with pytest.raises(KeyError):
                gz.fetch("nope", 0, 1)


def test_bgzf_writer_block_size_and_blocks_walk(tmp_path):
    from tredparse_b200 import bamio
    data = bytes(range(256)) * 40
    for bs in (1, 97, 0xFF00):
        w = bamio.BGZFWriter(str(tmp_path / "x.gz"), level=1, block_size=bs)
        w.write(data)
        w.close()
        blocks = bamio.bgzf_blocks(str(tmp_path / "x.gz"))
        sizes = [b[2] for b in blocks]
        assert sizes[-1] == 0 and sum(sizes) == len(data) and max(sizes) == min(bs, len(data))
        assert [b[1] for b in blocks] == list(np.cumsum([0] + sizes[:-1]))
        with gzip.open(str(tmp_path / "x.gz")) as fp:
            assert fp.read() == data
    for bs in (0, 0xFF01):
        with pytest.raises(ValueError):
            bamio.BGZFWriter(str(tmp_path / "y.gz"), block_size=bs)


# ---------------------------------------------------------------------------------------------------------------
# the tract scan on a BGZF file (host emulation of the device code) == the plain-text scan == the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width,crlf", WIDTHS)
@pytest.mark.parametrize("block", BLOCKS)
def test_emulated_scan_on_bgzf_equals_plain_and_the_oracle(tmp_path, width, crlf, block):
    contigs = _contigs(width, crlf)
    want = _oracle(width, crlf)
    for level in LEVELS:
        d = tmp_path / "l{}".format(level)
        d.mkdir()
        plain, gz = _pair(d, contigs, width, crlf, block, level)
        text = plain.tracts(MOTIFS, emulate=True)
        for step in (0, 2000, 700):                    # one step; many steps, blocks shared between steps
            got = gz.tracts(MOTIFS, step_bytes=step, emulate=True)
            assert _as_tuples(got) == want
            _check_plan(got, gz, step)
            assert got["stats"]["comp_bytes"] > 0 and got["stats"]["blocks"] > 0
            assert len(got["stats"]["step_read_ms"]) == len(got["stats"]["step_device_ms"]) == got["stats"]["steps"]
            if step == 0:
                assert {k: got["stats"][k] for k in STATS} == {k: text["stats"][k] for k in STATS}
        assert _as_tuples(text) == want
        assert text["stats"]["comp_bytes"] == 0 and text["stats"]["blocks"] == 0
        if block == 97:
            shared = gz.tracts(MOTIFS, step_bytes=700, emulate=True)["stats"]
            assert shared["blocks"] > len(gz.blocks) - 1   # some blocks are inflated by two steps


# ---------------------------------------------------------------------------------------------------------------
# errors
# ---------------------------------------------------------------------------------------------------------------
def _fai(fa):
    from tredparse_b200 import _lib
    names = list(fa.index)
    fai = np.zeros(len(names), dtype=_lib.FAI_ENTRY_DTYPE)
    for i, n in enumerate(names):
        fai[i] = fa.index[n]
    return fai


def _codes(motifs):
    from tredparse_b200.fasta import canonical_code
    return sorted({(len(m), canonical_code(m)) for m in motifs})


def test_plain_gzip_is_refused_and_bgzf_is_accepted(tmp_path):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    plain, gz = _pair(tmp_path, {"c1": "ACGT" * 30}, 60)
    assert gz.fetch("c1", 0, 8) == "ACGTACGT"
    pg = str(tmp_path / "plain.fa.gz")
    with gzip.open(pg, "wb") as fp:
        fp.write(b">c1\nACGT\n")
    with pytest.raises(ValueError, match="compressed.*bgzip"):
        Fasta(pg)
    # C: a gzip file that is not BGZF fails at framing
    with pytest.raises(_lib.TredswError, match=r"code -4\).*plain\.fa\.gz: not a BGZF block at offset 0"):
        _lib.ref_tracts(pg, _fai(plain), _codes(["AC"]), 3, 30, emulate=True)


def test_truncated_bgzf_files(tmp_path):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    contigs = _random_contigs(3, n=3, length=4000)
    plain, gz = _pair(tmp_path, contigs, 60, block=1000, level=6, fai=True)
    data = open(gz.path, "rb").read()
    k = len(gz.blocks) // 2
    coff = gz.blocks[k][0]
    # inside a block: the walk finds it
    cut = str(tmp_path / "cut.fa.gz")
    with open(cut, "wb") as fp:
        fp.write(data[:coff + 30])
    shutil.copyfile(gz.path + ".fai", cut + ".fai")
    with pytest.raises(IOError, match="truncated BGZF block at offset {}".format(coff)):
        Fasta(cut)
    with pytest.raises(_lib.TredswError, match=r"code -4\).*cut\.fa\.gz: truncated BGZF block at offset {}".format(coff)):
        _lib.ref_tracts(cut, _fai(gz), _codes(MOTIFS), 3, 30, emulate=True)
    # at a block boundary: every block is whole, and the .fai reaches past the inflated end
    with open(cut, "wb") as fp:
        fp.write(data[:coff])
    short = Fasta(cut)
    with pytest.raises(_lib.TredswError, match=r"code -4\).*past the end of the inflated text"):
        short.tracts(MOTIFS, emulate=True)
    with pytest.raises(_lib.TredswError, match=r"past the end of the inflated text"):
        short.tracts(MOTIFS, step_bytes=1000, emulate=True)
    with pytest.raises(ValueError, match="shorter than its index"):
        short.fetch("ctg2", 0, len(contigs["ctg2"]))
    assert short.fetch("ctg0", 0, 50) == contigs["ctg0"][:50].upper()


def test_corrupt_block(tmp_path):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    contigs = _random_contigs(4, n=3, length=4000)
    _, gz = _pair(tmp_path, contigs, 60, block=1000, level=6, fai=True)
    data = bytearray(open(gz.path, "rb").read())
    # a block in the middle of ctg1's text
    L, off, lb, lw = gz.index["ctg1"]
    k = next(i for i, (_, u, n) in enumerate(gz.blocks) if u > off + 1000)
    coff, uoff, isize = gz.blocks[k]
    bsize = gz.blocks[k + 1][0] - coff
    for at in (coff + 18 + 3, coff + 18 + (bsize - 26) // 2, coff + bsize - 12):  # DEFLATE data; framing intact
        bad = bytearray(data)
        bad[at] ^= 0x5A
        path = str(tmp_path / "bad.fa.gz")
        with open(path, "wb") as fp:
            fp.write(bytes(bad))
        shutil.copyfile(gz.path + ".fai", path + ".fai")
        fa = Fasta(path)
        assert fa.blocks == gz.blocks
        with pytest.raises(_lib.TredswError, match=r"code -4\).*bad\.fa\.gz: the BGZF block at offset {} ".format(coff)):
            fa.tracts(MOTIFS, emulate=True)
        with pytest.raises(_lib.TredswError, match="block at offset {} ".format(coff)):
            fa.tracts(MOTIFS, step_bytes=2000, emulate=True)
        i = (uoff + isize // 2 - off) // lw * lb                  # a base in the corrupt block
        with pytest.raises(IOError):
            fa.fetch("ctg1", i, i + 10)
        assert fa.fetch("ctg0", 0, 100) == contigs["ctg0"][:100].upper()
        assert fa.fetch("ctg2", 100, 300) == contigs["ctg2"][100:300].upper()
        os.remove(path + ".fai")                        # the index built in memory inflates the whole file
        with pytest.raises(IOError, match="bad.fa.gz"):
            Fasta(path)


def test_an_index_that_does_not_fit_the_inflated_text(tmp_path):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    contigs = {"a": "AC" * 200, "b": "CAG" * 100}
    plain, gz = _pair(tmp_path, contigs, 60, block=97)
    with open(gz.path + ".fai", "w") as fp:            # line width one byte short: a base position hits '\n'
        for n, (L, off, lb, lw) in plain.index.items():
            fp.write("{}\t{}\t{}\t{}\t{}\n".format(n, L, off, lb, lw - 1))
    with pytest.raises(_lib.TredswError, match=r"code -4\).*index does not fit"):
        Fasta(gz.path).tracts(["AC"], emulate=True)
    with open(gz.path + ".fai", "w") as fp:            # longer than the inflated text
        fp.write("a\t400\t3\t60\t61\nb\t100000\t{}\t60\t61\n".format(plain.index["b"][1]))
    with pytest.raises(_lib.TredswError, match=r"code -4\).*contig 1 .*past the end of the inflated text"):
        Fasta(gz.path).tracts(["AC"], emulate=True)


# ---------------------------------------------------------------------------------------------------------------
# strprofile loci on a bgzipped reference
# ---------------------------------------------------------------------------------------------------------------
def _loci_inputs(tmp_path):
    from test_ref_tracts import _loci_inputs as inputs
    from tredparse_b200 import simulate
    inputs(tmp_path)
    simulate.bgzip_fasta(str(tmp_path / "ref.fa"), str(tmp_path / "ref.fa.gz"), block_size=1000)


def _loci(tmp_path, fasta, *extra, env=ENV):
    return subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "loci", str(tmp_path / "out.tsv"),
                           "--fasta", str(tmp_path / fasta), "--profiles", str(tmp_path / "a.str_profile.json"),
                           *extra], cwd=str(tmp_path), env=env, capture_output=True, text=True)


def test_loci_on_a_bgzipped_reference(tmp_path):
    _loci_inputs(tmp_path)
    for fasta in ("ref.fa", "ref.fa.gz"):
        r = _loci(tmp_path, fasta, "--out", "{}.json".format(fasta))
        assert r.returncode == 0, r.stderr
    a, b = (open(str(tmp_path / "{}.json".format(f))).read() for f in ("ref.fa", "ref.fa.gz"))
    assert a == b and list(json.loads(a)) == ["c1_1001_GGGAA"]
    r = _loci(tmp_path, "ref.fa.gz", "--alts", "--out", str(tmp_path / "o.json"), env=dict(ENV, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "no CUDA device" in r.stderr and r.stdout == ""
    assert not os.path.exists(str(tmp_path / "o.json"))


# ---------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("width,crlf", WIDTHS)
@pytest.mark.parametrize("block", BLOCKS)
def test_gpu_kernels_on_bgzf_equal_the_emulation_and_plain_text(tmp_path, width, crlf, block):
    contigs = _contigs(width, crlf)
    want = _oracle(width, crlf)
    for level in LEVELS:
        d = tmp_path / "l{}".format(level)
        d.mkdir()
        plain, gz = _pair(d, contigs, width, crlf, block, level)
        for step in (0, 700):
            dev, emu, text = (gz.tracts(MOTIFS, step_bytes=step), gz.tracts(MOTIFS, step_bytes=step, emulate=True),
                              plain.tracts(MOTIFS, step_bytes=step))
            assert _as_tuples(dev) == _as_tuples(emu) == _as_tuples(text) == want
            keys = STATS + ("bytes", "comp_bytes", "blocks")
            assert {k: dev["stats"][k] for k in keys} == {k: emu["stats"][k] for k in keys}
            _check_plan(dev, gz, step)


@pytest.mark.gpu
def test_gpu_bgzf_equals_plain_on_100_mbp(tmp_path):
    from tredparse_b200 import simulate
    from tredparse_b200.fasta import Fasta
    path = _big_fasta(str(tmp_path / "big.fa"), 11, [41000000, 30000000, 20000000, 9000000, 777])
    plain, gz = Fasta(path), Fasta(simulate.bgzip_fasta(path, path + ".gz"))
    assert gz.index == plain.index
    a, b = plain.tracts(MOTIFS, step_bytes=16 << 20), gz.tracts(MOTIFS, step_bytes=16 << 20)
    assert np.array_equal(a["tracts"], b["tracts"]) and b["stats"]["tracts"] > 4000
    assert {k: a["stats"][k] for k in STATS} == {k: b["stats"][k] for k in STATS}
    assert b["stats"]["steps"] == 4 and b["stats"]["bases"] == 100000777
    _check_plan(b, gz, 16 << 20)
    assert b["stats"]["comp_bytes"] < os.path.getsize(gz.path) + 4 * 0x10000


@pytest.mark.gpu
def test_gpu_context_is_usable_after_a_corrupt_block(tmp_path):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    ctx = _lib.Context(0)
    contigs = _random_contigs(4, n=3, length=4000)
    plain, gz = _pair(tmp_path, contigs, 60, block=1000, level=6, fai=True)
    data = bytearray(open(gz.path, "rb").read())
    coff = gz.blocks[len(gz.blocks) // 2][0]
    data[coff + 40] ^= 0x5A
    with open(str(tmp_path / "bad.fa.gz"), "wb") as fp:
        fp.write(bytes(data))
    shutil.copyfile(gz.path + ".fai", str(tmp_path / "bad.fa.gz.fai"))
    with pytest.raises(_lib.TredswError, match=r"code -4\).*block at offset {} ".format(coff)):
        Fasta(str(tmp_path / "bad.fa.gz")).tracts(MOTIFS, ctx=ctx)
    want = plain.tracts(MOTIFS, emulate=True)
    for fa in (gz, plain):
        got = fa.tracts(MOTIFS, ctx=ctx)
        assert _as_tuples(got) == _as_tuples(want)


@pytest.mark.gpu
def test_gpu_discovery_workflow_with_a_bgzipped_reference(tmp_path, monkeypatch, capsys):
    from test_ref_tracts import SITES, _calls, _cohort
    from tredparse_b200 import simulate, strprofile
    bams = _cohort(tmp_path)
    simulate.bgzip_fasta(str(tmp_path / "ref.fa"), str(tmp_path / "ref.fa.gz"), block_size=4000)
    work = tmp_path / "w"
    assert strprofile.main(["profile", *bams, "--workdir", str(work)]) == 0
    profs = [str(work / "s{}.str_profile.json".format(s)) for s in range(4)]
    assert strprofile.main(["outliers", *profs, "--tsv", str(tmp_path / "out.tsv")]) == 0
    names = ["{}_{}_{}".format(c, pos + 1, u) for c, pos, u, _, _ in SITES]
    csv = tmp_path / "samples.csv"
    csv.write_text("".join("s{},{}\n".format(s, b) for s, b in enumerate(bams)))
    sites, calls = {}, {}
    for fasta in ("ref.fa", "ref.fa.gz"):
        run = tmp_path / ("run_" + fasta.replace(".", "_"))
        run.mkdir()
        monkeypatch.chdir(str(run))
        assert strprofile.main(["loci", str(tmp_path / "out.tsv"), "--fasta", str(tmp_path / fasta),
                                "--profiles", *profs, "--alts"]) == 0
        with open("sites/discovered.json") as fp:
            sites[fasta] = fp.read()
        calls[fasta] = _calls(csv, run / "calls", names + ["HD"])
    assert sites["ref.fa"] == sites["ref.fa.gz"]
    assert json.loads(sites["ref.fa.gz"])[names[0]]["alts"] == "c3:2000-2150|c3:6000-6100"
    assert calls["ref.fa"] == calls["ref.fa.gz"]
