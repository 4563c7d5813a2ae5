"""Build librla_b200.so in-tree with nvcc for sm_100a (no JIT cache, no fallback).

    python -m rla4mor_b200._build            # build if stale
    python -m rla4mor_b200._build --force
"""
import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librla_b200.so")
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--shared", "-Xptxas", "-v",
    "-Wno-deprecated-gpu-targets",
]
# NumPy's Gaussian stream is reproduced bit for bit only without contracted multiply-adds
FILE_FLAGS = {"mt19937.cu": ["--fmad=false", "-Xcompiler", "-ffp-contract=off"]}


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: librla_b200.so cannot be built (there is no CPU fallback)")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + \
        [os.path.join(os.path.dirname(HERE), "include", "rla_b200.h")]
    return any(os.path.getmtime(p) > t for p in deps)


def build_library(force=False, verbose=False):
    """Compile every .cu under csrc/ into one shared library.  Returns the path."""
    if not force and not is_stale():
        return LIB
    objs = []
    objdir = os.path.join(HERE, "csrc", "_obj")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    env = dict(os.environ)
    # the image exports CC=/opt/gcc/bin/gcc, whose specs lack what nvcc's host pass needs
    ccbin = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else None
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if (not force and os.path.exists(obj) and os.path.getmtime(obj) > os.path.getmtime(src)
                and all(os.path.getmtime(obj) > os.path.getmtime(h)
                        for h in glob.glob(os.path.join(CSRC, "*.cuh")) +
                        [os.path.join(os.path.dirname(HERE), "include", "rla_b200.h")])):
            continue
        cmd = [_nvcc()] + [f for f in NVCC_FLAGS if f != "--shared"] + FILE_FLAGS.get(os.path.basename(src), []) + \
            ["-c", src, "-o", obj]
        if ccbin:
            cmd += ["-ccbin", ccbin]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)))
    log = []
    for src, pr in procs:
        out, _ = pr.communicate()
        log.append(out)
        if pr.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [_nvcc(), "--shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    if ccbin:
        cmd += ["-ccbin", ccbin]
    subprocess.run(cmd, check=True)
    with open(os.path.join(objdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        sys.stderr.write("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
