"""Build libnabo_b200.so in-tree with nvcc for sm_100a (no torch extension, no JIT cache)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnabo_b200.so")
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(os.path.dirname(HERE), "include", "nabo_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into one shared library.  Returns its path."""
    if not force and not _stale():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libnabo_b200.so must be prebuilt (it ships in-tree)")
    objdir = os.path.join(HERE, "csrc", "_obj")
    os.makedirs(objdir, exist_ok=True)
    common = [nvcc, *ARCH_FLAGS, "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr", "-Xptxas", "-v" if verbose else "-O3"]
    common += os.environ.get("NABO_NVCC_EXTRA", "").split()      # development switches (e.g. -DNABO_CBS_PROF)
    objs = []
    procs = []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or _obj_stale(obj, src):
            procs.append((src, subprocess.Popen(common + ["-c", src, "-o", obj],
                                                stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out.decode())
            raise RuntimeError("nvcc failed on %s" % src)
        if verbose:
            sys.stderr.write(out.decode())
    tmp = LIB + ".tmp"
    subprocess.check_call([nvcc, *ARCH_FLAGS, "-shared", "-o", tmp, *objs, "-lcuda"])
    os.replace(tmp, LIB)
    return LIB


def _obj_stale(obj: str, src: str) -> bool:
    t = os.path.getmtime(obj)
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
           [os.path.join(os.path.dirname(HERE), "include", "nabo_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
