#!/usr/bin/env python
"""
Golden calls on a simulated whole-sample BAM, for tests/test_gpu_reference.py:

    python tests/golden/make_oracle_bam_fixture.py      -> tests/golden/oracle_sample_bam.json

The BAM is sample 3 of tredparse_b200.simulate (cohort seed, +-2 kb windows at NAMES, contigs of t001.mini.bam).
The calls are those of the CPU oracle (oracle/genotype_oracle.py: evidence_oracle + likelihood_oracle on the
sw_oracle.c aligner), which tests/test_reference_pinned.py holds to the outputs of tredparse 0.7.8 itself.  The
SHA-1 over the BAM's records (not its compressed bytes, which depend on the zlib build) catches a simulator that no
longer writes the same reads.
"""
import hashlib
import json
import logging
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

NAMES = ["HD", "DM1", "FXS", "FRDA", "SCA10", "ULD", "OPMD", "AR"]
SAMPLE, FLANK = 3, 2000
OUT = os.path.join(HERE, "oracle_sample_bam.json")


def write_sample(path, repo):
    """The simulated BAM (+ .bai) at `path` -> the truth {tred: alleles}."""
    from tredparse_b200 import simulate, bamio
    sam = bamio.AlignmentFile(os.path.join(HERE, "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    return simulate.write_sample_bam(path, repo, NAMES, refs, SAMPLE, flank=FLANK)


def records_sha1(path):
    from tredparse_b200 import bamio
    h = hashlib.sha1()
    for r in bamio.AlignmentFile(path).fetch():
        h.update(repr((r.query_name, r.flag, r.reference_id, r.reference_start, r.mapping_quality, r.cigartuples,
                       r.next_reference_id, r.next_reference_start, r.template_length, r.query_sequence)).encode())
    return h.hexdigest()


def jsonable(x):
    if isinstance(x, dict):
        return {str(k): jsonable(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [jsonable(v) for v in x]
    if hasattr(x, "item"):
        return x.item()
    return x


def oracle_calls(path, repo):
    """tred.run's per-sample pre-steps (gender, read length), then the oracle's calls of every locus."""
    import numpy as np
    from oracle import genotype_oracle
    from tredparse_b200 import bamio, tred as T
    pre = T.presteps(path, repo, NAMES, logging.getLogger("fixture"))
    with open(os.path.join(ROOT, "tredparse_b200", "data", "models.json")) as fp:
        md = json.load(fp)
    step = {int(k): np.array(v) for k, v in md["step_size_by_period"].items()}
    for i in range(6, 18):
        step[i] = step[6]
    sam = bamio.AlignmentFile(path)
    calls = {}
    for n in NAMES:
        c, _, _ = genotype_oracle.genotype_locus(sam, repo[n], pre["readLen"], step, md["stutter_weights"],
                                                 gender=pre["inferredGender"])
        calls[n] = jsonable(c)
    return pre, calls


def main():
    import tempfile
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "s.bam")
        truth = write_sample(path, repo)
        pre, calls = oracle_calls(path, repo)
        doc = {"source": "CPU oracle (oracle/genotype_oracle.py) on simulated sample {} (+-{} bp windows)".format(SAMPLE, FLANK),
               "names": NAMES, "truth": jsonable(truth), "records_sha1": records_sha1(path),
               "presteps": jsonable(pre), "calls": calls}
    with open(OUT, "w") as fp:
        json.dump(doc, fp, sort_keys=True)
    print(OUT, os.path.getsize(OUT))


if __name__ == "__main__":
    main()
