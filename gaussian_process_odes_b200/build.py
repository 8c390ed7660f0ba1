"""Builds ``libgpode_b200.so`` (the C-ABI CUDA library of include/gpode_b200.h) in-tree with nvcc for sm_100a.

    python -m gaussian_process_odes_b200.build [--force] [--verbose]

The library has no torch / Python dependency: plain ``nvcc -shared``. Objects go to ``csrc/build/`` (git-ignored),
the shared library next to this file so that it travels to the GPU box with the repo snapshot.
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJDIR = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libgpode_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-I", INCLUDE]

# (source, extra defines, object name)
UNITS = [("pack.cu", [], "pack.o"), ("param_grad.cu", [], "param_grad.o"), ("whiten.cu", [], "whiten.o"), ("whiten_blocked.cu", [], "whiten_blocked.o"),
         ("integrate.cu", [], "integrate.o"), ("dopri5.cu", [], "dopri5.o"), ("probe.cu", [], "probe.o"), ("side_terms.cu", [], "side_terms.o"), ("large_d.cu", [], "large_d.o"), ("large_umma.cu", [], "large_umma.o"), ("large_bwd.cu", [], "large_bwd.o"), ("large_rffb.cu", [], "large_rffb.o"), ("large_dopri5.cu", [], "large_dopri5.o"), ("large_shoot.cu", [], "large_shoot.o")] + \
        [("integrate_d.cu", ["-DGPODE_D=%d" % d], "integrate_d%d.o" % d) for d in range(1, 9)] + \
        [("dopri5_d.cu", ["-DGPODE_D=%d" % d], "dopri5_d%d.o" % d) for d in range(1, 9)]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; the gpode_b200 CUDA library cannot be built")
    return exe


def _newest_source_mtime():
    m = os.path.getmtime(os.path.join(INCLUDE, "gpode_b200.h"))
    for f in os.listdir(CSRC):
        if f.endswith((".cu", ".cuh", ".h")):
            m = max(m, os.path.getmtime(os.path.join(CSRC, f)))
    return max(m, os.path.getmtime(os.path.abspath(__file__)))


def _compile(unit, verbose):
    src, defs, obj = unit
    objp = os.path.join(OBJDIR, obj)
    cmd = [_nvcc()] + NVCC_FLAGS + defs + ["-c", os.path.join(CSRC, src), "-o", objp]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(objp + ".log", "w") as fh:
        fh.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr[-4000:]))
    if verbose:
        print("compiled", obj)
    return objp


def build(force=False, verbose=False):
    """Compile (if stale) and return the path of the shared library."""
    units = [u for u in UNITS if os.path.exists(os.path.join(CSRC, u[0]))]
    newest = _newest_source_mtime()
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= newest:
        return LIB
    os.makedirs(OBJDIR, exist_ok=True)
    todo, objs = [], []
    for u in units:
        objp = os.path.join(OBJDIR, u[2])
        objs.append(objp)
        if force or not os.path.exists(objp) or os.path.getmtime(objp) < newest:
            todo.append(u)
    workers = max(1, min(len(todo), os.cpu_count() or 1))
    if todo:
        with concurrent.futures.ThreadPoolExecutor(workers) as ex:
            list(ex.map(lambda u: _compile(u, verbose), todo))
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr[-4000:])
    if verbose:
        print("linked", LIB)
    return LIB


def ptxas_report():
    """(kernel, registers, spill bytes) from the last build's ptxas -v logs -- used by DESIGN.md / tests."""
    import re
    out = []
    for f in sorted(os.listdir(OBJDIR)) if os.path.isdir(OBJDIR) else []:
        if not f.endswith(".log"):
            continue
        s = open(os.path.join(OBJDIR, f)).read()
        for name, sst, sld, regs in re.findall(
                r"Compiling entry function '(\S+)' for 'sm_100a'\n.*?\n.*?bytes stack frame, (\d+) bytes spill stores, "
                r"(\d+) bytes spill loads\n.*?Used (\d+) registers", s):
            out.append((f[:-6], name, int(regs), int(sst) + int(sld)))
    return out


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv or True)
    print(p)
