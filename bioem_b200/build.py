"""Build libbioem_b200.so (CUDA kernels + C ABI) in-tree for sm_100a with nvcc.

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU
box with the working tree.  The fused likelihood kernel is instantiated in one
translation unit per supported image edge (csrc/lik_instance.inl) so that the
variants compile in parallel."""
from __future__ import annotations

import concurrent.futures as cf
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libbioem_b200.so")
SOURCES = ["bioem_b200.cu", "host_prep.cpp"]
HEADERS = ["bioem_kernels.cuh", "generic_kernels.cuh", "render_kernels.cuh", "fft_regs.cuh", "lik_instance.inl",
           os.path.join("..", "..", "include", "bioem_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CFLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
          "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "-Xptxas", "-v"]


def sizes() -> list[int]:
    src = open(os.path.join(CSRC, "bioem_b200.cu")).read()
    out = []
    for macro in ("BIOEM_SIZES_TUNED", "BIOEM_SIZES_AUTO"):
        m = re.search(r"#define " + macro + r"\(X\)(.*)", src)
        out += [int(x) for x in re.findall(r"X\((\d+)\)", m.group(1))]
    return out


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def _compile(args):
    name, cmd = args
    r = subprocess.run(cmd, capture_output=True, text=True)
    return name, r.returncode, " ".join(cmd) + "\n" + r.stdout + r.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    jobs = []
    objs = []
    for s in SOURCES:
        o = os.path.join(OBJ, s + ".o")
        objs.append(o)
        jobs.append((s, [NVCC] + CFLAGS + ["-c", os.path.join(CSRC, s), "-o", o]))
    for n in sizes():
        o = os.path.join(OBJ, f"lik_{n}.o")
        objs.append(o)
        jobs.append((f"lik_{n}", [NVCC] + CFLAGS + [f"-DBIOEM_N={n}", "-x", "cu", "-c",
                                                    os.path.join(CSRC, "lik_instance.inl"), "-o", o]))
    log = []
    failed = []
    with cf.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        for name, rc, out in ex.map(_compile, jobs):
            log.append(f"==== {name} (rc={rc})\n{out}")
            if rc != 0:
                failed.append(name)
    if not failed:
        r = subprocess.run([NVCC, "-shared", "-ccbin", "/usr/bin/g++", "-o", LIB] + objs, capture_output=True, text=True)
        log.append("==== link\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            failed.append("link")
    with open(os.path.join(HERE, "build.log"), "w") as f:
        f.write("\n".join(log))
    if failed:
        sys.stderr.write("\n".join(log)[-8000:])
        raise RuntimeError(f"nvcc failed building libbioem_b200.so: {failed}")
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
