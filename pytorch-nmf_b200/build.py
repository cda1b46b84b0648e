"""Build libnmf_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python pytorch-nmf_b200/build.py [--force] [--verbose]

The output (pytorch-nmf_b200/lib/libnmf_b200.so) is git-ignored but travels to the GPU box.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libnmf_b200.so")
SOURCES = ["capi.cu", "simt_nmf.cu", "update.cu", "nmfd.cu", "tc_nmf.cu", "tc_nmfd.cu", "sparse_nmf.cu", "project.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build libnmf_b200.so")


def source_hash():
    """sha256 over every file the library is compiled from (csrc/*, include/nmf_b200.h), first 16 hex digits.  Compiled
    into the library (nmfb200_build_info) so a test can prove the .so on the GPU box was built from these sources."""
    import hashlib
    h = hashlib.sha256()
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC)) + [os.path.join(HERE, "..", "include", "nmf_b200.h")]
    for f in files:
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(HERE, "..", "include", "nmf_b200.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a into one shared library.  Returns the library path."""
    if not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    stamp = source_hash()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + [f'-DNMFB200_SRC_HASH="{stamp}"'] + (["-Xptxas", "-v"] if verbose else []) + [
            "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link of libnmf_b200.so failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
