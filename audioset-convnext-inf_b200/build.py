"""Builds csrc/*.cu into libacx.so (in-tree, sm_100a only) with a plain nvcc call.

The shared library is git-ignored but travels to the GPU box with the gpurun snapshot."""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libacx.so")
STAMP = os.path.join(HERE, ".libacx.stamp")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
         "-shared", "-cudart", "static"]


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest():
    h = hashlib.sha256()
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC))
    files.append(os.path.join(os.path.dirname(HERE), "include", "acx.h"))
    for f in files:
        h.update(f.encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile if sources changed; returns the path of libacx.so."""
    dig = _digest()
    if not force and os.path.isfile(LIB) and os.path.isfile(STAMP) and open(STAMP).read().strip() == dig:
        return LIB
    if not os.path.isfile(NVCC):
        raise RuntimeError(f"nvcc not found at {NVCC}; cannot build libacx.so")
    objs = []
    procs = []
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    compile_flags = [f for f in FLAGS if f not in ("-shared",)]
    for src in _sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = [NVCC, "-c", src, "-o", obj] + [f for f in compile_flags if f not in ("-cudart", "static")]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {os.path.basename(src)} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libacx.so")
    link = [NVCC, "-shared", "-o", LIB, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"] + objs
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("nvcc link failed for libacx.so")
    with open(STAMP, "w") as fh:
        fh.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
