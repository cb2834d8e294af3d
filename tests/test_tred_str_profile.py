"""`tred.py --str-profile`: the one GPU scan of each sample serves its catalogue calls and its STR profile
(<samplekey>.str_profile.json, the dict of strprofile.profile).  Indexed BAMs are scanned instead of read by the
indexed ingest, unindexed BAMs and streams keep their one scan; under --gpus N one rank profiles each sample.

The cohort: whole-sample BAMs with background pairs, catalogue loci (FXS is X-linked, so gender is inferred; two
samples carry chrY reads) and planted expansions away from the catalogue (simulate.expansion_records), with and
without mismapped in-repeat reads and MQ tags.  CPU tests cover the rank rule, the parent's merge, the command line and
the routing of prepare_chunk through the host emulation of the device code; the `gpu` tests run tred.main."""
import contextlib
import gzip
import json
import logging
import os
import shutil
import subprocess
import sys
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
NAMES = ["HD", "DM1", "FXS", "SCA1"]
# (planted expansion (motif, contig index, units) or None, MQ tags, mismapped fraction, chrY reads)
SAMPLES = [(("AAGGG", 1, 200), True, 0.3, False), (None, False, 0.0, True), (("ATTC", 2, 90), False, 0.0, False),
           (None, True, 0.2, True)]
PLANTED = {("AAGGG", "s0"), ("AATG", "s2")}           # (canonical motif, sample) of the planted expansions


def _refs():
    from tredparse_b200 import bamio
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    return refs


def _write_sample(path, s):
    """sample s of SAMPLES as an indexed BAM whose @RG SM is s<s> (the sample key of stdin)"""
    from tredparse_b200 import bamio, simulate
    from tredparse_b200.bam_parser import BamDepth
    from tredparse_b200.meta import TREDsRepo
    planted, mq_tags, mismap, male = SAMPLES[s]
    repo, refs = TREDsRepo(), _refs()
    tid = {n: i for i, (n, _) in enumerate(refs)}
    rng = np.random.default_rng(s)
    recs = []
    for k in range(200):                                        # background pairs over the first contigs
        t = int(rng.integers(0, 3))
        p = int(rng.integers(1000, refs[t][1] - 1000))
        recs += simulate.expansion_records(t, p, "AC", 0, cov=2, flank=400, seed=s * 1000 + k, tag="bg{}_".format(k),
                                           mq_tags=mq_tags)
    for li, name in enumerate(NAMES):
        t = repo[name]
        alleles = (int(rng.integers(10, 25)), int(rng.integers(15, 40)))      # (shorter than a read: no IRRs)
        recs += simulate.locus_records(t, tid[t.chr], alleles, 150, 6.0, seed=10 * s + li, tag="l{}_".format(li),
                                       flank=1000)
    if planted:
        motif, t, units = planted
        recs += simulate.expansion_records(t, refs[t][1] // 3, motif, units, cov=10, seed=50 + s, tag="far",
                                           mq_tags=mq_tags, mismap_fraction=mismap,
                                           mismap_to=(0, 1000, refs[0][1] - 1000) if mismap else None)
    elif mismap:                                                # mismapped IRRs of a short expansion: shared noise
        recs += simulate.expansion_records(2, refs[2][1] // 2, "CAG", 60, cov=6, seed=70 + s, tag="cag", mq_tags=mq_tags,
                                           mismap_fraction=mismap, mismap_to=(0, 1000, refs[0][1] - 1000))
    if male:                                                    # ~15x over the chrY regions of the gender inference
        for c, a, b in BamDepth.y_regions("hg38"):
            n = 15 * (b - a) // 100
            for k, p in enumerate(sorted(rng.integers(a, b - 100, n).tolist())):
                seq = "".join("ACGT"[x] for x in rng.integers(0, 4, 100))
                recs.append(bamio.AlignedSegment("y{}_{}".format(a, k), 0, tid[c], p, 60, [(0, 100)], -1, -1, 0, seq))
    text = ("@HD\tVN:1.4\tSO:coordinate\n" + "".join("@SQ\tSN:{}\tLN:{}\n".format(n, l) for n, l in refs)
            + "@RG\tID:g\tSM:s{}\n".format(s))
    bamio.write_bam(path, refs, simulate.coordinate_sort(recs), header_text=text, aux=True)
    return path


@pytest.fixture(scope="module")
def cohort(tmp_path_factory):
    """{"indexed": [paths], "unindexed": [copies without .bai]}"""
    d = tmp_path_factory.mktemp("tred_str_profile")
    idx = [_write_sample(str(d / "s{}.bam".format(s)), s) for s in range(len(SAMPLES))]
    os.makedirs(str(d / "noindex"))
    un = []
    for p in idx:
        un.append(str(d / "noindex" / os.path.basename(p)))
        shutil.copy(p, un[-1])
    return {"indexed": idx, "unindexed": un}


def _read(path):
    with open(path, "rb") as fp:
        return fp.read()


def _tasks(paths, names=NAMES):
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    return [("s{}".format(i), p, repo, list(names), 300, False, False, True, True, "INFO") for i, p in enumerate(paths)]


def _csv(path, paths):
    with open(path, "w") as fp:
        for i, p in enumerate(paths):
            fp.write("s{},{}\n".format(i, p))
    return path


def _tred_args(workdir):
    out = ["--workdir", str(workdir)]
    for n in NAMES:
        out += ["--tred", n]
    return out


def _cli(args, cwd, **kw):
    env = dict(os.environ, PYTHONPATH=ROOT)
    return subprocess.run([sys.executable, "-m", "tredparse_b200.tred"] + args, cwd=cwd, env=env, capture_output=True,
                          timeout=900, **kw)


def _vcf_lines(path):
    with gzip.open(path, "rt") as fp:
        return [l for l in fp.read().splitlines() if not l.startswith("##fileDate")]


def _outputs(workdir, key):
    """(JSON text, VCF lines without ##fileDate, profile dict or None) of one sample"""
    w = str(workdir)
    prof = os.path.join(w, key + ".str_profile.json")
    with open(os.path.join(w, key + ".json")) as fp:
        js = fp.read()
    return js, _vcf_lines(os.path.join(w, key + ".tred.vcf.gz")), (json.load(open(prof)) if os.path.exists(prof) else None)


def _want_profile(path, key, bam=None):
    """strprofile.profile of the file == the oracle's, after a JSON round trip; bam set to what the run names"""
    from tredparse_b200 import strprofile
    from oracle import irr_oracle
    got = json.loads(json.dumps(strprofile.profile(path, sample=key)))
    ref = json.loads(json.dumps(irr_oracle.profile(path, sample=key)))
    assert got == ref
    if bam is not None:
        got["bam"] = bam
    return got


@contextlib.contextmanager
def _fifo(path, data):
    """a named pipe at `path` that a thread writes `data` into once a reader opens it"""
    os.mkfifo(path)

    def feed():
        try:
            fd = os.open(path, os.O_WRONLY)
        except OSError:
            return
        try:
            view = memoryview(data)
            for i in range(0, len(data), 1 << 16):
                os.write(fd, view[i:i + (1 << 16)])
        except BrokenPipeError:
            pass
        finally:
            os.close(fd)
    t = threading.Thread(target=feed, daemon=True)
    t.start()
    try:
        yield path
    finally:
        if t.is_alive():
            try:
                os.close(os.open(path, os.O_RDONLY | os.O_NONBLOCK))
            except OSError:
                pass
        t.join(timeout=60)
        os.unlink(path)


@contextlib.contextmanager
def _piped(data):
    """the read end of a pipe a thread writes `data` into, as /dev/fd/N"""
    r, w = os.pipe()

    def feed():
        try:
            view, i = memoryview(data), 0
            while i < len(data):
                i += os.write(w, view[i:i + (1 << 16)])
        except BrokenPipeError:
            pass
        finally:
            os.close(w)
    t = threading.Thread(target=feed, daemon=True)
    t.start()
    try:
        yield "/dev/fd/{}".format(r)
    finally:
        os.close(r)
        t.join(timeout=60)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the rank rule, the parent's merge, the command line
# ---------------------------------------------------------------------------------------------------------------
def test_profile_rank_owns_most_loci_ties_to_the_lowest_rank():
    from tredparse_b200 import tred as T
    keys = [(0, "A"), (0, "B"), (0, "C"), (1, "A"), (1, "B"), (2, "A"), (2, "B"), (2, "C"), (2, "D")]
    owner = np.array([1, 0, 1, 2, 1, 3, 2, 2, 3], dtype=np.int32)
    # sample 0: rank 1 owns 2; sample 1: ranks 1 and 2 own 1 each (tie: 1); sample 2: ranks 2 and 3 own 2 each (2);
    # sample 3: no locus
    assert T.profile_ranks(owner, keys, 4) == [1, 1, 2, None]
    assert T.profile_ranks(np.zeros(len(keys), np.int32), keys, 3) == [0, 0, 0]
    # on a real deal: every profile rank owns a locus of its sample, and the rule is the same on every call
    tasks = _tasks(["a.bam", "b.bam", "c.bam"], names=["HD", "DM1", "FXS", "SCA1", "SCA2"])
    owner, keys = T.deal(tasks, 3)
    ranks = T.profile_ranks(owner, keys, 3)
    assert ranks == T.profile_ranks(*T.deal(tasks, 3), 3)
    for si, r in enumerate(ranks):
        mine = [o for (s, _), o in zip(keys, owner.tolist()) if s == si]
        assert r in mine and mine.count(r) == max(mine.count(o) for o in set(mine))
        assert r == min(o for o in set(mine) if mine.count(o) == mine.count(r))


def _part(key, calls, prof=None, error=None):
    from tredparse_b200 import tred as T
    r = {"samplekey": key, "bam": key + ".bam", "tredCalls": dict(calls)}
    if prof is not None:
        r[T.STR_PROFILE] = prof
    if error:
        r["error"] = error
    return r


def test_part_merge_waits_for_all_loci_and_the_profile():
    from tredparse_b200 import tred as T
    # three samples of 2 loci each; sample 0 profiled by rank 1, sample 1 by rank 0, sample 2 by rank 1
    m = T.PartMerge([2, 2, 2], profile_rank=[1, 0, 1])
    assert m.add(0, 0, _part("a", {"HD.1": 1}), 1) == []                       # sample 0: its profile part is missing
    assert m.add(0, 1, _part("b", {"HD.1": 3}, prof={"sample": "b"}), 1) == []   # sample 1 is held: sample 0 first
    assert m.add(1, 1, _part("b", {"DM1.1": 4}), 1) == []
    out = m.add(1, 0, _part("a", {"DM1.1": 2}, prof={"sample": "a"}), 1)      # the profile part arrives last
    assert [r["samplekey"] for r in out] == ["a", "b"]
    assert out[0] == {"samplekey": "a", "bam": "a.bam", "tredCalls": {"HD.1": 1, "DM1.1": 2}, T.STR_PROFILE: {"sample": "a"}}
    assert out[1][T.STR_PROFILE] == {"sample": "b"} and out[1]["tredCalls"] == {"HD.1": 3, "DM1.1": 4}
    # all the loci are in, but the part of the profile rank is not: held until it comes (a failed scan: no profile)
    assert m.add(0, 2, _part("c", {"HD.1": 5, "DM1.1": 6}), 2) == []
    out = m.add(1, 2, _part("c", {}, error="RuntimeError('boom')"), 0)
    assert out == [{"samplekey": "c", "bam": "c.bam", "tredCalls": {"HD.1": 5, "DM1.1": 6}}]
    assert m.rest() == []
    # without profiles: released on the loci alone, as before
    m = T.PartMerge([1, 2])
    assert m.add(1, 1, _part("b", {"x": 1}), 2) == []
    assert [r["samplekey"] for r in m.add(0, 0, _part("a", {"y": 1}), 1)] == ["a", "b"]
    # a sample whose parts never all came is released at the end
    m = T.PartMerge([2, 1], profile_rank=[0, 0])
    assert m.add(0, 1, _part("b", {"z": 1}, prof={}), 1) == []
    assert [r["samplekey"] for r in m.rest()] == ["b"]


def test_str_profile_refused_without_the_gpu_scan(tmp_path):
    """TREDSW_GPU_INGEST=0: an argument error before anything is read (stdin stays open and empty: a read would
    block)"""
    r, w = os.pipe()
    try:
        res = subprocess.run([sys.executable, "-m", "tredparse_b200.tred", "-", "--workdir", str(tmp_path / "w"),
                              "--tred", "HD", "--str-profile"], cwd=str(tmp_path), stdin=r, capture_output=True,
                             timeout=300, env=dict(os.environ, PYTHONPATH=ROOT, TREDSW_GPU_INGEST="0"))
    finally:
        os.close(r)
        os.close(w)
    assert res.returncode != 0 and b"--str-profile" in res.stderr and b"TREDSW_GPU_INGEST=0" in res.stderr, res.stderr
    assert not os.listdir(str(tmp_path / "w"))


def _fake_run_chunks(seen):
    from tredparse_b200 import tred as T

    def fake(task_args, only=None, chunk=None, isolate=False, str_profile=False):
        seen.append(([a[0] for a in task_args], str_profile))
        for a in task_args:
            r = {"samplekey": a[0], "bam": a[1], "tredCalls": {"inferredGender": "Female", "depthY": 0.0, "readLen": 150}}
            if str_profile:
                r[T.STR_PROFILE] = {"sample": a[0], "profile": {}}
            yield r
    return fake


def test_emit_writes_the_profile_beside_the_json_and_no_output_writes_nothing(tmp_path, monkeypatch):
    from tredparse_b200 import tred as T
    seen = []
    monkeypatch.setattr(T, "run_chunks", _fake_run_chunks(seen))
    csv = _csv(str(tmp_path / "samples.csv"), ["/nonexistent/a.bam", "/nonexistent/b.bam"])
    w = tmp_path / "w"
    T.main([csv, "--workdir", str(w), "--tred", "HD", "--str-profile"])
    assert seen == [(["s0", "s1"], True)]
    for k in ("s0", "s1"):
        js = json.loads((w / (k + ".json")).read_text())
        assert T.STR_PROFILE not in js and set(js) == {"samplekey", "bam", "tredCalls"}
        assert json.loads((w / (k + ".str_profile.json")).read_text()) == {"sample": k, "profile": {}}
    T.main([csv, "--workdir", str(tmp_path / "w0"), "--tred", "HD"])
    assert seen[-1] == (["s0", "s1"], False) and not list((tmp_path / "w0").glob("*.str_profile.json"))
    T.main([csv, "--workdir", str(tmp_path / "none"), "--tred", "HD", "--str-profile", "--no-output"])
    assert seen[-1] == (["s0", "s1"], True) and os.listdir(str(tmp_path / "none")) == []


def test_checkexists_skips_the_sample_and_its_profile(tmp_path, monkeypatch):
    from tredparse_b200 import tred as T
    seen = []
    monkeypatch.setattr(T, "run_chunks", _fake_run_chunks(seen))
    csv = _csv(str(tmp_path / "samples.csv"), ["/nonexistent/a.bam", "/nonexistent/b.bam"])
    w = tmp_path / "w"
    w.mkdir()
    (w / "s0.json").write_text("{}\n")
    T.main([csv, "--workdir", str(w), "--tred", "HD", "--str-profile", "--checkexists"])
    assert seen == [(["s1"], True)]
    assert sorted(os.listdir(str(w))) == ["s0.json", "s1.json", "s1.str_profile.json", "s1.tred.vcf.gz"]
    assert (w / "s0.json").read_text() == "{}\n"
    assert "such a sample gets no STR profile" in " ".join(T.set_argparse().format_help().split())


# ---------------------------------------------------------------------------------------------------------------
# CPU: prepare_chunk's routing, through the host emulation of the device code
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture
def emulated(monkeypatch):
    """no device: the GPU ingest and the scan run their host emulation (a None context)"""
    from tredparse_b200 import _lib
    monkeypatch.setattr(_lib, "default_context", lambda device=None: None)


def _prepared(args, **kw):
    from tredparse_b200 import tred as T
    state = T.prepare_chunk(args, **kw)
    _, out, items, where, device_batch = state
    ev = {k: (it[1], it[2], it[3], it[4].reads.tobytes(), it[4].roff.tobytes(), tuple(it[4].names),
              np.asarray(it[4].global_lens).tobytes(), np.asarray(it[4].target_lens).tobytes())
          for k, it in zip(where, items)}
    if device_batch is not None:
        device_batch.close()
    return out, ev


def test_emulated_indexed_sample_is_scanned_once_with_the_same_evidence(cohort, emulated, monkeypatch):
    """--str-profile on indexed BAMs: one scan per sample, no indexed ingest, no host reader; evidence, gender, depthY
    and read length equal the run without the flag; the profile equals the oracle's"""
    from tredparse_b200 import tred as T, ingest, strprofile
    from oracle import irr_oracle
    args = _tasks(cohort["indexed"])
    out0, ev0 = _prepared(args)
    assert {o["tredCalls"]["inferredGender"] for o in out0} == {"Male", "Female"}
    assert all(T.STR_PROFILE not in o for o in out0)

    def forbidden(*a, **k):
        raise AssertionError("read by something else than the sample's one scan")
    scans = []
    real_scan, real_batch, real_gender = ingest.scan_sample, ingest.IngestBatch, T.infer_gender

    def counted(*a, **k):
        b = real_scan(*a, **k)
        scans.append((b.stats()["records"], k.get("irr") is not None))
        return b
    monkeypatch.setattr(ingest, "scan_sample", counted)
    monkeypatch.setattr(ingest, "IngestBatch", forbidden)
    monkeypatch.setattr(T, "ingest_loci", forbidden)
    monkeypatch.setattr(T, "infer_gender", forbidden)
    monkeypatch.setattr(strprofile, "profile", forbidden)
    out1, ev1 = _prepared(args, str_profile=True)
    assert len(scans) == len(args) and all(n > 1000 and irr for n, irr in scans)
    assert ev1 == ev0 and len(ev0) == len(args) * len(NAMES)
    for o0, o1, (key, path) in zip(out0, out1, [(a[0], a[1]) for a in args]):
        assert o1["tredCalls"] == o0["tredCalls"]
        assert o1[T.STR_PROFILE] == irr_oracle.profile(path, sample=key)
    # the cohort table ranks the planted expansions first
    regions = [r for r in strprofile.outliers([o[T.STR_PROFILE] for o in out1]) if r["contig"] != "-"]
    assert {(r["motif"], r["top_sample"]) for r in regions[:2]} == PLANTED
    # one bool per sample: only the second sample is scanned, the others go through the indexed ingest
    scans.clear()
    monkeypatch.setattr(ingest, "IngestBatch", real_batch)
    monkeypatch.setattr(T, "infer_gender", real_gender)
    out2, ev2 = _prepared(args, str_profile=[False, True, False, False])
    assert len(scans) == 1 and ev2 == ev0
    assert [T.STR_PROFILE in o for o in out2] == [False, True, False, False]


def test_emulated_failed_scan_keeps_the_calls_route_and_logs_the_missing_profile(cohort, emulated, tmp_path, caplog):
    """a truncated unindexed file: the loci go to the host reader as without the flag, no profile, an error names the
    sample and the scan status"""
    from tredparse_b200 import tred as T
    data = _read(cohort["unindexed"][0])
    bad = str(tmp_path / "cut.bam")
    with open(bad, "wb") as fp:
        fp.write(data[:len(data) * 2 // 3])
    args = _tasks([bad])
    out0, ev0 = _prepared(args)
    with caplog.at_level(logging.ERROR, logger="tredparse_b200.tred"):
        out1, ev1 = _prepared(args, str_profile=True)
    assert ev1 == ev0 and out1[0]["tredCalls"] == out0[0]["tredCalls"] and T.STR_PROFILE not in out1[0]
    msgs = [r.getMessage() for r in caplog.records if "no STR profile" in r.getMessage()]
    assert msgs and "`s0`" in msgs[0] and "status" in msgs[0]


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _run_main(argv):
    from tredparse_b200 import tred as T
    cwd = os.getcwd()
    try:
        T.main(argv)
    finally:
        os.chdir(cwd)


@pytest.mark.gpu
def test_gpu_str_profile_on_files_and_a_fifo(cohort, tmp_path):
    """indexed BAMs, their unindexed copies and FIFOs listed in a CSV: with --str-profile, every sample's profile is
    strprofile.profile's (== the oracle's) and its JSON and VCF are those of the run without the flag; the calls
    are those of the indexed run"""
    base = None                                     # the calls of the indexed run without the flag
    for kind in ("indexed", "unindexed", "fifo"):
        outs = {}
        for flag in (False, True):
            w = tmp_path / "{}_{}".format(kind, int(flag))
            with contextlib.ExitStack() as es:
                if kind == "fifo":
                    paths = [es.enter_context(_fifo(str(tmp_path / "f{}.bam".format(i)), _read(p)))
                             for i, p in enumerate(cohort["indexed"])]
                else:
                    paths = cohort[kind]
                csv = _csv(str(tmp_path / "{}_{}.csv".format(kind, int(flag))), paths)
                _run_main([csv] + _tred_args(w) + (["--str-profile"] if flag else []))
            outs[flag] = {"s{}".format(i): _outputs(w, "s{}".format(i)) for i in range(len(paths))}
        if base is None:
            base = {k: json.loads(o[0])["tredCalls"] for k, o in outs[False].items()}
        for i, src in enumerate(cohort["indexed"]):
            key = "s{}".format(i)
            (j0, v0, p0), (j1, v1, p1) = outs[False][key], outs[True][key]
            assert p0 is None and j1 == j0 and v1 == v0, (kind, key)
            js = json.loads(j1)
            assert p1 == _want_profile(src, key, bam=js["bam"]), (kind, key)
            assert p1["sample"] == key and js["tredCalls"] == base[key], (kind, key)
    assert {base[k]["inferredGender"] for k in base} == {"Male", "Female"}


@pytest.mark.gpu
def test_gpu_stdin_is_read_once_for_calls_and_profile(cohort, tmp_path):
    """`... | python -m tredparse_b200.tred - --str-profile`: JSON and VCF of the run without the flag, the file's profile
    (bam `-`); the outliers step takes it next to profiles from `strprofile profile`"""
    src = cohort["indexed"][0]
    outs = {}
    for flag in (False, True):
        w = tmp_path / "stdin_{}".format(int(flag))
        res = _cli(["-"] + _tred_args(w) + (["--str-profile"] if flag else []), str(tmp_path), input=_read(src))
        assert res.returncode == 0, res.stderr[-3000:]
        outs[flag] = _outputs(w, "s0")
    (j0, v0, p0), (j1, v1, p1) = outs[False], outs[True]
    assert p0 is None and j1 == j0 and v1 == v0
    assert p1 == _want_profile(src, "s0", bam="-")
    env = dict(os.environ, PYTHONPATH=ROOT)
    others = tmp_path / "others"
    subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "profile", *cohort["indexed"][1:], "--workdir",
                    str(others)], check=True, env=env, cwd=ROOT)
    files = [str(tmp_path / "stdin_1" / "s0.str_profile.json")] + sorted(str(p) for p in others.glob("*.str_profile.json"))
    res = subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "outliers", *files], check=True, env=env,
                         cwd=ROOT, capture_output=True, text=True)
    regions = [l.split("\t") for l in res.stdout.splitlines()[1:] if not l.startswith("-\t")]
    assert {(r[3], r[4]) for r in regions[:2]} == PLANTED


@pytest.mark.gpu
def test_gpu_pipe_sample_needs_no_second_read(cohort, monkeypatch):
    """run_chunks on a pipe: the calls and the profile come from its one scan; a second read of it finds nothing"""
    from tredparse_b200 import tred as T, ingest, strprofile
    src = cohort["indexed"][2]
    want = list(T.run_chunks(_tasks([src])))[0]
    want_prof = _want_profile(src, "s0")

    def forbidden(*a, **k):
        raise AssertionError("the stream was read a second time")
    monkeypatch.setattr(strprofile, "profile", forbidden)
    with _piped(_read(src)) as path:
        got = list(T.run_chunks(_tasks([path]), str_profile=True))[0]
        with pytest.raises(IOError):
            ingest.BamIngest.stream(path)
    prof = got.pop(T.STR_PROFILE)
    assert "error" not in got and got["tredCalls"] == want["tredCalls"]
    assert json.loads(json.dumps(prof)) == dict(want_prof, bam=path)


@pytest.mark.gpu
def test_gpu_indexed_sample_goes_through_one_scan_and_no_indexed_ingest(cohort, monkeypatch):
    from tredparse_b200 import tred as T, ingest
    args = _tasks(cohort["indexed"])
    want = [r["tredCalls"] for r in T.run_chunks(args)]

    def forbidden(*a, **k):
        raise AssertionError("the indexed ingest or the host reader was used")
    monkeypatch.setattr(ingest, "IngestBatch", forbidden)
    monkeypatch.setattr(T, "ingest_loci", forbidden)
    scans = []
    real = ingest.scan_sample

    def counted(*a, **k):
        b = real(*a, **k)
        scans.append(b.stats()["records"])
        return b
    monkeypatch.setattr(ingest, "scan_sample", counted)
    got = list(T.run_chunks(args, str_profile=True))
    assert len(scans) == len(args) and all(n > 1000 for n in scans)
    for r, w, (key, path) in zip(got, want, [(a[0], a[1]) for a in args]):
        assert r["tredCalls"] == w
        assert json.loads(json.dumps(r[T.STR_PROFILE])) == _want_profile(path, key)


@pytest.mark.gpu
def test_gpu_corrupt_unindexed_file_gets_calls_and_no_profile(cohort, tmp_path, caplog):
    data = _read(cohort["unindexed"][1])
    bad = tmp_path / "in"
    bad.mkdir()
    path = str(bad / "cut.bam")
    with open(path, "wb") as fp:
        fp.write(data[:len(data) * 2 // 3])
    csv = _csv(str(tmp_path / "cut.csv"), [path])
    _run_main([csv] + _tred_args(tmp_path / "w0"))
    with caplog.at_level(logging.ERROR, logger="tredparse_b200.tred"):
        _run_main([csv] + _tred_args(tmp_path / "w1") + ["--str-profile"])
    j0, v0, p0 = _outputs(tmp_path / "w0", "s0")
    j1, v1, p1 = _outputs(tmp_path / "w1", "s0")
    assert p0 is None and p1 is None and j1 == j0 and v1 == v0
    assert not list((tmp_path / "w1").glob("*.str_profile.json"))
    assert any("`s0`" in r.getMessage() and "status" in r.getMessage() and "no STR profile" in r.getMessage()
               for r in caplog.records)


def _two_gpus():
    try:
        import torch
        return torch.cuda.device_count() >= 2
    except Exception:
        return False


@pytest.mark.gpu
def test_gpu_two_ranks_profile_each_sample_once(cohort, tmp_path, monkeypatch):
    if not _two_gpus():
        pytest.skip("needs two visible GPUs")
    from tredparse_b200 import tred as T
    written = []
    real = T.write_str_profile

    def counted(key, prof):
        written.append(key)
        return real(key, prof)
    monkeypatch.setattr(T, "write_str_profile", counted)
    paths = cohort["indexed"][:2] + cohort["unindexed"][2:]
    csv = _csv(str(tmp_path / "s.csv"), paths)
    runs = {}
    for name, extra in (("g1p", ["--gpus", "1", "--str-profile"]), ("g2", ["--gpus", "2"]),
                        ("g2p", ["--gpus", "2", "--str-profile"])):
        _run_main([csv] + _tred_args(tmp_path / name) + extra)
        runs[name] = {"s{}".format(i): _outputs(tmp_path / name, "s{}".format(i)) for i in range(len(paths))}
    assert sorted(written) == sorted(["s{}".format(i) for i in range(len(paths))] * 2)
    for k in runs["g2p"]:
        assert runs["g2p"][k][0] == runs["g2"][k][0] and runs["g2p"][k][1] == runs["g2"][k][1]
        assert runs["g2p"][k][2] == runs["g1p"][k][2] is not None
