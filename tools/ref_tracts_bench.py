#!/usr/bin/env python
"""The reference tract scan (Fasta.tracts, tredsw_ref_tracts) on a whole synthetic genome: a seeded FASTA with the
contig sizes of hg38 scaled to --gbp, 60-base lines, half of every contig soft-masked (lowercase) in 4 KiB blocks, an
N run at either end of every contig and one in its middle (~3 % of its length), and planted tracts of the motifs it
scans for.  The motifs are those of 20 loci of periods 2 to 20 (what `strprofile loci --alts` asks for after a cohort
with that many discovered loci).

One context, then --reps + 1 calls: the first call on its own (pinned buffers allocated, modules loaded) and the best
of the later ones.  The card's name, power limit and max SM clock are read in the same run.  The file is written to a
temporary directory, never into the repository, and is read from the page cache (the run writes it just before): a
cold-cache read and a real reference genome are not measured.

--bgzip adds a second arm: a BGZF copy of the same genome (64 KiB blocks at zlib level 6, as `bgzip` writes it; the
blocks are compressed on every host core, since they are independent) with the same .fai, whose blocks the scan
inflates on the GPU.  The two arms alternate call by call, and each reports its first call and the best of the later
ones.  The synthetic genome (uniform random bases) compresses less well than hg38, whose repeats and soft-masking
give DEFLATE more to work with: the compressed-to-text ratio here is not hg38's.

--max-interruption N also plants interrupted tracts (one every 50 kb, from a second seeded stream, so the rest of the
genome is unchanged: 6 to 40 copies of a motif with 1 to 3 substitutions, insertions or deletions) and splits every
format into two arms that alternate call by call: the pure rule and the chain rule with interruptions of up to N bases
at purity 9 / 10 (DESIGN §4.5.1).  Each arm reports its tracts and how many of them are chains.  Uniform random
sequence rarely chains by chance, so those counts say nothing about hg38.

    python tools/ref_tracts_bench.py [--gbp 3.1] [--reps 3] [--step-mib 256] [--bgzip] [--max-interruption N]
                                     [--out profiles/r3_ref_tracts_bench.json]
(without --out the result line is only printed)
"""
import argparse
import concurrent.futures
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HG38_MBP = [248.96, 242.19, 198.30, 190.21, 181.54, 170.81, 159.35, 145.14, 138.39, 133.80, 135.09, 133.28, 114.36,
            107.04, 101.99, 90.34, 83.26, 80.37, 58.62, 64.44, 46.71, 50.82, 156.04, 57.23]
NAMES = ["chr{}".format(i) for i in range(1, 23)] + ["chrX", "chrY"]
MOTIFS = ["AC", "AT", "AG", "CAG", "AAG", "ATC", "AAAG", "AATG", "AAGGG", "AAAAT", "AACCCT", "AAGGCC", "AGCGGCG",
          "AACCTGG", "ACCGGAGCG", "AGGTTCCAGC", "AAGGTACCGTT", "ACGTTGCAAGCT", "TGCTTACCGTCAA",
          "GATCCAGTTAGCCTGAAAGT"]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception as e:
        return "unknown ({})".format(e)


def interrupted_tract(rng):
    """a tract of 6 to 40 copies of a motif with 1 to 3 interruptions: a substitution, an insertion of 1 to 3 bases
    or a deletion of one base"""
    from tredparse_b200.simulate import interrupted_tract as planted
    u = MOTIFS[int(rng.integers(len(MOTIFS)))]
    n = int(rng.integers(6, 41))
    edits = []
    for c in sorted(set(int(x) for x in rng.integers(1, n, int(rng.integers(1, 4))))):
        x = rng.random()
        if x < 0.5:
            edits.append((c, "sub", "ACGT"["ACGT".index(u[0]) ^ 1]))
        elif x < 0.8:
            edits.append((c, "ins", "".join("ACGT"[int(b)] for b in rng.integers(0, 4, int(rng.integers(1, 4))))))
        else:
            edits.append((c, "del", 1))
    return planted(u, n, edits)


def write_genome(path, gbp, seed=0, width=60, interrupted=False):
    rng = np.random.default_rng(seed)
    irng = np.random.default_rng(seed + 1)
    lut = np.frombuffer(b"ACGT", np.uint8)
    scale = gbp * 1e3 / sum(HG38_MBP)
    total, fai = 0, []
    with open(path, "wb") as fp:
        for name, mbp in zip(NAMES, HG38_MBP):
            L = int(mbp * 1e6 * scale)
            s = lut[rng.integers(0, 4, L, dtype=np.uint8)]
            for _ in range(L // 50000):                     # planted tracts, 3 to 40 copies
                u = MOTIFS[int(rng.integers(len(MOTIFS)))]
                t = np.frombuffer((u * int(rng.integers(3, 41))).encode(), np.uint8)
                a = int(rng.integers(0, L - len(t)))
                s[a:a + len(t)] = t
            for _ in range(L // 50000 if interrupted else 0):
                t = np.frombuffer(interrupted_tract(irng).encode(), np.uint8)
                a = int(irng.integers(0, L - len(t)))
                s[a:a + len(t)] = t
            nb = L // 4096                                  # soft-masking: half of the 4 KiB blocks in lowercase
            blocks = s[:nb * 4096].reshape(nb, 4096)
            blocks[rng.random(nb) < 0.5] += 32
            for a, n in ((0, 10000), (L // 2, L // 33), (L - 10000, 10000)):
                s[a:a + n] = ord("N")
            fp.write(">{}\n".format(name).encode())
            fai.append("{}\t{}\t{}\t{}\t{}\n".format(name, L, fp.tell(), width, width + 1))
            n = (L + width - 1) // width
            body = np.full((n, width + 1), ord("\n"), np.uint8)
            pad = np.full(n * width, ord("\n"), np.uint8)
            pad[:L] = s
            body[:, :width] = pad.reshape(n, width)
            fp.write(body.tobytes()[:L + n])
            total += L
    with open(path + ".fai", "w") as fp:
        fp.writelines(fai)
    return total


def bgzip(src, dst, level=6, block=0xFF00, chunk_blocks=1024):
    """a BGZF copy of src (the .fai copied too: its offsets are those of the inflated text), blocks compressed on a
    thread pool (zlib releases the GIL)"""
    from tredparse_b200.bamio import bgzf_block
    with open(src, "rb") as fi, open(dst, "wb") as fo, \
            concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 1) as pool:
        while True:
            data = fi.read(block * chunk_blocks)
            if not data:
                break
            parts = [data[i:i + block] for i in range(0, len(data), block)]
            for b in pool.map(lambda x: bgzf_block(x, level), parts):
                fo.write(b)
        fo.write(bgzf_block(b"", level))
    shutil.copyfile(src + ".fai", dst + ".fai")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbp", type=float, default=3.1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--step-mib", type=int, default=256)
    ap.add_argument("--bgzip", action="store_true", help="also scan a BGZF copy of the genome, the arms alternating")
    ap.add_argument("--max-interruption", type=int, default=0,
                    help="plant interrupted tracts and add a chain arm per format (1 to 20)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    g = a.max_interruption
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    ctx = _lib.default_context()
    d = tempfile.mkdtemp(prefix="ref_tracts_bench_")
    try:
        path = os.path.join(d, "genome.fa")
        t0 = time.time()
        bases = write_genome(path, a.gbp, interrupted=g > 0)
        t_write = time.time() - t0
        paths = {"text": path}
        if a.bgzip:
            t0 = time.time()
            bgzip(path, path + ".gz")
            t_bgzip = time.time() - t0
            paths["bgzf"] = path + ".gz"
        fas = {f: Fasta(p) for f, p in paths.items()}
        # arm -> (format, max_interrupt)
        arms_g = {f: (f, 0) for f in paths} if not g else \
            {"{}_{}".format(f, r): (f, x) for f in paths for r, x in (("pure", 0), ("chain", g))}
        calls = {arm: [] for arm in arms_g}
        for _ in range(a.reps + 1):                     # the arms alternate call by call
            for arm, (f, x) in arms_g.items():
                t0 = time.perf_counter()
                r = fas[f].tracts(MOTIFS, step_bytes=a.step_mib << 20, ctx=ctx, max_interrupt=x)
                calls[arm].append((time.perf_counter() - t0, r))
        for arm, (_, x) in arms_g.items():              # every call of one rule gives the same tracts
            ref = calls[next(b for b, (_, y) in arms_g.items() if y == x)][0][1]
            for _, r in calls[arm]:
                assert np.array_equal(r["tracts"], ref["tracts"]) and np.array_equal(r["segments"], ref["segments"]), arm

        def summary(wall, res):
            s = res["stats"]
            return {"wall_s": round(wall, 4), "lib_ms_total": round(s["ms_total"], 2),
                    "text_GB_per_s": round(s["bytes"] / wall / 1e9, 3),
                    "host_read_ms_sum": round(sum(s["step_read_ms"]), 2),
                    "device_ms_sum": round(sum(s["step_device_ms"]), 2)}

        def arm_result(arm):
            first, later = calls[arm][0], calls[arm][1:]
            best = min(later, key=lambda c: c[0]) if later else first
            st = best[1]["stats"]
            out = {"file_bytes": os.path.getsize(paths[arms_g[arm][0]]), "steps": st["steps"], "text_bytes": st["bytes"],
                   "comp_bytes": st["comp_bytes"], "blocks": st["blocks"], "invalid_bases": st["invalid_bases"],
                   "tracts": st["tracts"]}
            if g:                                       # counts only: the per-tract segments stay out of the card
                out.update(max_interrupt=arms_g[arm][1], chains=int((best[1]["segments"] > 1).sum()))
            return dict(out, **{"first_call": summary(*first), "best_later_call": summary(*best),
                    "later_walls_s": [round(w, 4) for w, _ in later],
                    "per_step_best": [{"read_ms": round(x, 2), "device_ms": round(y, 2)}
                                      for x, y in zip(st["step_read_ms"], st["step_device_ms"])]})

        head = {"card": card(), "gbp": a.gbp, "bases": bases, "write_s": round(t_write, 1), "motifs": len(MOTIFS),
                "step_mib": a.step_mib}
        cache = "warm (files written in the same run); cold cache not measured"
        if g:
            arms = {arm: arm_result(arm) for arm in arms_g}
            out = dict({"bench": "ref_tracts_chain"}, **head, max_interruption=g, purity=[9, 10], arms=arms,
                       chain_note="uniform random sequence rarely chains by chance: the chain counts come from the "
                                  "planted interrupted tracts and say nothing about hg38", page_cache=cache)
            if a.bgzip:
                out.update(bgzip_s=round(t_bgzip, 1))
        elif not a.bgzip:
            out = dict({"bench": "ref_tracts"}, **head, **arm_result("text"), page_cache=cache.replace("files", "file"))
            del out["comp_bytes"], out["blocks"]
        else:
            arms = {arm: arm_result(arm) for arm in paths}
            out = dict({"bench": "ref_tracts_bgzf"}, **head, bgzip_s=round(t_bgzip, 1), arms=arms,
                       comp_ratio=round(arms["bgzf"]["file_bytes"] / arms["text"]["file_bytes"], 4),
                       comp_ratio_note="uniform random bases with soft-masking and N runs: not hg38's ratio",
                       tracts_equal_across_arms=True, page_cache=cache)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fp:
            json.dump(out, fp, indent=1)
            fp.write("\n")


if __name__ == "__main__":
    main()
