"""Builds libpn_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python code-adaptive-prob-ode-solvers_b200/build.py [--force]

One translation unit per problem family, compiled in parallel; the shared library is git-ignored.
The kernel headers are also embedded in the library (build/pn_jit_sources.inc), for the run-time
compilation of user-defined vector fields (csrc/pn_jit.cu); NVRTC is linked statically (README).
"""

import concurrent.futures
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libpn_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-std=c++17", "-O3", "-lineinfo",
    # fp64 contract: no implicit contraction; every FMA in the kernels is an explicit fma()
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true",
    "-Xcompiler", "-fPIC",
    "-diag-suppress", "177,128",
]  # fmt: skip


# NVRTC and its device-code compiler, linked into the library (README, "User-defined vector fields")
NVRTC_LIBS = ["-lnvrtc_static", "-lnvrtc-builtins_static", "-lnvptxcompiler_static", "-lpthread", "-ldl"]
JIT_SOURCES = os.path.join(OBJ, "pn_jit_sources.inc")
_DELIM = "pn_src"


def write_jit_sources(headers):
    """build/pn_jit_sources.inc: every csrc/*.cuh as {file name, text}; rewritten only when it changes."""
    parts = []
    for h in sorted(headers):
        text = open(h, encoding="utf-8").read()
        if f'){_DELIM}"' in text:
            raise RuntimeError(f"{h} contains the raw-string delimiter ){_DELIM}\"")
        parts.append(f'{{"{os.path.basename(h)}", R"{_DELIM}({text}){_DELIM}"}},\n')
    body = "struct JitSource {\n  const char* name;\n  const char* text;\n};\nconst JitSource kJitSources[] = {\n" + "".join(parts) + "};\n"
    old = open(JIT_SOURCES, encoding="utf-8").read() if os.path.exists(JIT_SOURCES) else None
    if old != body:
        with open(JIT_SOURCES, "w", encoding="utf-8") as f:
            f.write(body)


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    hdrs = glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h"))
    hdrs += [os.path.join(HERE, "..", "include", "pn_b200.h"), os.path.abspath(__file__)]
    os.makedirs(OBJ, exist_ok=True)
    write_jit_sources(glob.glob(os.path.join(CSRC, "*.cuh")))
    dep_time = _newest(hdrs)
    jobs = []
    objs = []
    for s in srcs:
        o = os.path.join(OBJ, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(dep_time, os.path.getmtime(s)):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        extra = os.environ.get("PN_EXTRA_NVCC_FLAGS", "").split()
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-I", OBJ, "-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return s, r.returncode, r.stdout + r.stderr

    if jobs:
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for s, rc, out in ex.map(compile_one, jobs):
                if verbose or rc:
                    sys.stderr.write(out)
                if rc:
                    raise RuntimeError(f"nvcc failed on {s}")
    if jobs or not os.path.exists(LIB) or os.path.getmtime(LIB) < _newest(objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"] + NVRTC_LIBS
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
