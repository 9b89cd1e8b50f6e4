"""Build libpgdbg.so (sm_100a) in-tree with nvcc.

    python -m pangenome_b200.build [--force]

The library travels to the GPU box with the repo snapshot (it is git-ignored,
not gpurun-ignored); nothing is JIT-compiled at run time.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpgdbg.so")
SOURCES = ["common.cu", "fasta_pack.cu", "dbg_table.cu", "path_graph.cu", "partition.cu", "region_build.cu", "multisplit.cu", "compact_build.cu", "host_io.cu", "microbench.cu", "mcl.cu", "bgzf_inflate.cu", "fastq_pack.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.isfile(os.path.join(CSRC, s))]


def needs_build():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "pgdbg.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "_build"), exist_ok=True)
    for src in _sources():
        obj = os.path.join(HERE, "_build", os.path.basename(src)[:-3] + ".o")
        cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd)))
        objs.append(obj)
    for cmd, p in procs:
        if p.wait() != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
