"""Build libaligntools_b200.so in-tree with nvcc for sm_100a (no JIT cache: the built
library travels to the GPU box with the repo snapshot)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libaligntools_b200.so")
ROOT = os.path.dirname(os.path.dirname(HERE))
HOST_DIR = os.path.join(ROOT, "host")
HOST_SOURCES = ["alignTools.c", "at_fasta.c"]
HOST_HEADERS = ["at_fasta.h"]
CLI = os.path.join(ROOT, "bin", "alignTools")
FASTA_DUMP = os.path.join(ROOT, "bin", "at_fasta_dump")
SOURCES = ["at_runtime.cu", "at_shim.cu"]
HEADERS = ["at_kernels.cuh", "at_cell.cuh", "at_band.h", "at_ptr_layout.h", "at_plan.h", "at_fill_affine.cuh", "at_wavefront.cuh", "at_devmem.h", "at_pipeline.inl", os.path.join("..", "..", "..", "include", "aligntools_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unused-function", "--threads", "0"]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def _host_stale() -> bool:
    if not os.path.exists(CLI) or not os.path.exists(FASTA_DUMP):
        return True
    t = min(os.path.getmtime(CLI), os.path.getmtime(FASTA_DUMP))
    deps = [os.path.join(HOST_DIR, s) for s in HOST_SOURCES + HOST_HEADERS + ["at_fasta_dump.c"]] + [LIB, os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_host(force: bool = False) -> str:
    """The C host (bin/alignTools): the reference's CLI over the C-ABI library, plus the FASTA
    reader's test driver.  Plain gcc; the binary finds the library through an $ORIGIN rpath."""
    if not force and not _host_stale():
        return CLI
    os.makedirs(os.path.dirname(CLI), exist_ok=True)
    cflags = ["-std=gnu11", "-O2", "-g", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", HOST_DIR]
    subprocess.run(["gcc"] + cflags + [os.path.join(HOST_DIR, s) for s in HOST_SOURCES] +
                   ["-o", CLI, "-L", HERE, "-laligntools_b200", "-lz", "-Wl,-rpath,$ORIGIN/../aligntools/c_b200"], check=True)
    subprocess.run(["gcc"] + cflags + [os.path.join(HOST_DIR, "at_fasta_dump.c"), os.path.join(HOST_DIR, "at_fasta.c")] +
                   ["-o", FASTA_DUMP, "-lz"], check=True)
    return CLI


def build(force: bool = False, verbose: bool = False) -> str:
    lib = _build_lib(force, verbose)
    build_host(force)
    return lib


def build_variant(name: str, defines: list) -> str:
    """A/B builds: the library compiled with extra -D flags into lib_<name>.so beside the product library (load it with
    AT_LIB_PATH); used by tools/ab_*.sh to time kernel variants in one GPU call."""
    out = os.path.join(HERE, f"lib_{name}.so")
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(CSRC, s.replace(".cu", f".{name}.o"))
        cmd = ["nvcc"] + NVCC_FLAGS + [f"-D{d}" for d in defines] + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for cmd, p in procs:
        outp, _ = p.communicate()
        if p.returncode:
            sys.stderr.write(outp.decode())
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    subprocess.run(["nvcc", "-arch=sm_100a", "-shared", "-o", out] + objs + ["-lpthread"], check=True)
    return out


def _build_lib(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(CSRC, s.replace(".cu", ".o"))
        cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out.decode())
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    cmd = ["nvcc", "-arch=sm_100a", "-shared", "-o", LIB] + objs + ["-lpthread"]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
