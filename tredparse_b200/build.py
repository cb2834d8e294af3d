"""
Build libtredsw.so (the sm_100a CUDA library behind include/tredsw.h) in-tree with nvcc.

    python -m tredparse_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the resulting tredparse_b200/libtredsw.so is git-ignored but
travels with the source tree to the GPU box.
"""
import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libtredsw.so")
SOURCES = ["capi.cu", "sw_pairs.cu", "sw_family.cu", "grid.cu", "cohort.cu", "ingest.cpp", "bgzf_gpu.cu"]
INCLUDE = os.path.abspath(os.path.join(HERE, "..", "include"))
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def up_to_date():
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    # every file under csrc/ and include/ is a dependency (a header list kept by hand went stale once)
    deps = [p for p in glob.glob(os.path.join(CSRC, "*")) + glob.glob(os.path.join(INCLUDE, "*"))
            if not p.endswith(".o")] + [os.path.abspath(__file__)]
    return all(os.path.getmtime(d) <= t for d in deps)


def build(force=False, verbose=False, outdir=None, defines=()):
    """Build the library in-tree, or with outdir: objects and library in that directory (always rebuilt), compiled
    with the macros in defines (e.g. TREDSW_PHASE_CLOCKS for tools/phase_clock_bench.py)."""
    lib = os.path.join(outdir, "libtredsw.so") if outdir else OUT
    if not outdir and not force and up_to_date():
        return OUT
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(outdir or CSRC, os.path.splitext(s)[0] + ".o")
        cmd = [nvcc_path(), "-O3", "-std=c++17", *ARCH, "-lineinfo", "--extended-lambda", "-Xcompiler", "-fPIC",
               *["-D" + d for d in defines], "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for s, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode:
            sys.stderr.write(out.decode("utf-8", "replace"))
        if pr.returncode:
            raise RuntimeError("nvcc failed on {}".format(s))
    subprocess.check_call([nvcc_path(), *ARCH, "-shared", "-o", lib] + objs + ["-lz"])
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
