"""In-tree build of librala_b200.so (hand-written sm_100a kernels + the C ABI).

    python -m rala_b200.build [--verbose]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the
gpurun snapshot.  sm_100a only: no other -gencode, no PTX fallback for other architectures.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librala_b200.so")
SOURCES = ["classify.cu", "containment.cu", "graph_build.cu", "transitive.cu", "api.cu", "fabric.cu", "multi_api.cu", "frontend.cu", "paf.cu", "piles.cu", "reads.cu", "bgzf.cu", "gzip.cu"]
HEADERS = ["common.cuh", "lists.cuh", "kernels.h", "session.h", "fabric.cuh", "bgzf.cuh", "deflate.cuh", os.path.join("..", "..", "include", "rala_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _compile(lib: str, objdir: str, defines, verbose: bool) -> str:
    objs, procs = [], []
    os.makedirs(objdir, exist_ok=True)
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + list(defines) + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    os.makedirs(os.path.dirname(lib), exist_ok=True)
    link = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs
    subprocess.run(link, check=True)
    return lib


def build(verbose: bool = False, force: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    return _compile(LIB, os.path.join(HERE, "build"), [], verbose)


# A/B libraries for bench.py --ab, built by `python -m rala_b200.build --variants` into rala_b200/variants/.
# An optimisation under trial goes behind a compile-time switch that is on by default, and gets an entry here: VARIANTS
# maps a library name to the switch that library turns off (-D<macro>=0), TUNINGS to other -D settings of a tunable.
# The commit that settles the experiment removes both the switch and its entry, so every kernel keeps one code path.
# bench.py --ab also times `prev`, the parent commit's library built by profiles/build_prev.sh.
VARIANTS: dict = {}
TUNINGS: dict = {}
VARIANT_DIR = os.path.join(HERE, "variants")


def variant_path(name: str) -> str:
    return os.path.join(VARIANT_DIR, f"librala_b200_{name}.so")


def build_variants(verbose: bool = False):
    out = {}
    for name, macro in VARIANTS.items():
        out[name] = _compile(variant_path(name), os.path.join(HERE, "build", name), [f"-D{macro}=0"], verbose)
    for name, defines in TUNINGS.items():
        out[name] = _compile(variant_path(name), os.path.join(HERE, "build", name), defines, verbose)
    return out


if __name__ == "__main__":
    print(build(verbose="--verbose" in sys.argv, force=True))
    if "--variants" in sys.argv:
        for k, v in build_variants().items():
            print(k, v)
