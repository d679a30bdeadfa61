"""Build libsocp_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libsocp_b200.so")
# the parity build of SURVEY.md section 8(d): the same sources without FMA contraction (-fmad=false), to report the
# trajectory parity of both builds side by side (selected at run time with SOCP_LIB=<path>, tools/parity_builds.py)
SO_NOFMA = os.path.join(HERE, "libsocp_b200_nofma.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def sources():
    out = [os.path.join(HERE, "..", "include", "socp_b200.h")]
    for f in sorted(os.listdir(CSRC)):
        out.append(os.path.join(CSRC, f))
    return out


def stale(so=SO):
    if not os.path.exists(so):
        return True
    t = os.path.getmtime(so)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force=False, verbose=False, nofma=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo ... -> socp_b200/libsocp_b200.so
    (nofma=True: the -fmad=false parity build -> socp_b200/libsocp_b200_nofma.so)"""
    so = SO_NOFMA if nofma else SO
    if not force and not stale(so):
        return so
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-fmad=false"] if nofma else []) + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", so, os.path.join(CSRC, "api.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libsocp_b200.so")
    if verbose:
        print(r.stderr)
    return so


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, nofma="--nofma" in sys.argv))
