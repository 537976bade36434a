"""Build libphifem_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

    python -m phifem_b200.build [--force] [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libphifem_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"] + ARCH
# tags.cu restates the reference's exact ==1.0 comparisons: no FMA contraction there
SOURCES = [("capi.cu", []), ("tags.cu", ["-fmad=false"]), ("assemble.cu", []), ("assemble_rows.cu", []), ("assemble_tiles.cu", []), ("assemble_pk.cu", []), ("assemble_quad.cu", []), ("assemble_elasticity.cu", []), ("symbolic.cu", []), ("rows_plan.cu", []), ("solve.cu", []), ("peer.cu", [])]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, n) for n in os.listdir(CSRC) if n.endswith((".cu", ".cuh"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "phifem_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objs = []
    for name, extra in SOURCES:
        obj = os.path.join(CSRC, name[:-3] + ".o")
        cmd = [nvcc, "-c", os.path.join(CSRC, name), "-o", obj] + COMMON + extra
        if verbose:
            cmd += ["-Xptxas", "-v"]
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
        objs.append(obj)
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ARCH
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
