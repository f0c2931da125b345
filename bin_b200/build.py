"""Build libbin_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbin_b200.so")
SOURCES = ["conv_igemm.cu", "rdb_tail.cu", "aux_kernels.cu", "wgrad.cu", "metrics.cu", "train_data.cu", "api.cu"]
HEADERS = ["common.cuh", "internal.h", os.path.join("..", "..", "include", "bin_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest(sources=None, headers=None, extra=()) -> str:
    h = hashlib.sha256()
    for f in (sources or SOURCES) + (headers or HEADERS):
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(list(NVCC_FLAGS) + list(extra)).encode())
    return h.hexdigest()


TOOLS_LIB = os.path.join(HERE, "libbin_b200_tools.so")
TOOLS_SOURCES = SOURCES + ["tools_kernels.cu"]
TOOLS_HEADERS = HEADERS + ["tools_abi.h"]


def up_to_date(lib: str = LIB) -> bool:
    stamp = lib + ".sha256"
    tools = lib == TOOLS_LIB
    return (os.path.exists(lib) and os.path.exists(stamp) and
            open(stamp).read().strip() == _digest(TOOLS_SOURCES if tools else SOURCES, TOOLS_HEADERS if tools else HEADERS,
                                                  ["-DBIN_B200_TOOLS"] if tools else []))


def build_tools(force: bool = False, verbose: bool = False) -> str:
    """libbin_b200_tools.so: the product sources with -DBIN_B200_TOOLS (role-timeline hooks, per-call option re-reads)
    plus the microbenchmark kernels.  Used by tools/*.py only (BIN_B200_LIB selects it); never by the package."""
    return build(force, verbose, tools=True)


def build(force: bool = False, verbose: bool = False, tools: bool = False) -> str:
    LIB = TOOLS_LIB if tools else globals()["LIB"]
    SOURCES = TOOLS_SOURCES if tools else globals()["SOURCES"]
    extra = ["-DBIN_B200_TOOLS"] if tools else []
    stamp = LIB + ".sha256"
    dig = _digest(SOURCES, TOOLS_HEADERS if tools else HEADERS, extra)
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", "_tools.o" if tools else ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log.append(r.stdout)
    if r.returncode != 0:
        sys.stderr.write("\n".join(log))
        raise RuntimeError("link failed")
    with open(os.path.join(HERE, "build", "nvcc_tools.log" if tools else "nvcc.log"), "w") as fh:
        fh.write("\n".join(log))
    with open(stamp, "w") as fh:
        fh.write(dig)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True, tools="--tools" in sys.argv))
