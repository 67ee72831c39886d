"""Build recipe of libespm_b200.so (hand-written sm_100a CUDA behind a C ABI).

    python -m espm_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The library is built IN-TREE (espm_b200/lib/) so that it travels
with the repository snapshot to the GPU box; it is git-ignored.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
LIBNAME = "libespm_b200.so"
LIBPATH = os.path.join(LIBDIR, LIBNAME)

SOURCES = ["api.cu", "stream_f32f32.cu", "stream_f32f64.cu", "stream_f64f64.cu", "stream_u8f32.cu", "stream_u16f32.cu",
           "small_f32.cu", "small_f64.cu", "ingest.cu"]
HEADERS = ["common.cuh", "xpass.cuh", "xpass_inst.cuh", "small.cuh", "small_inst.cuh", "ingest.cuh", "ingest_decl.h",
           "fitstats.cuh", "hinfo.cuh", "winfo.cuh", "resid.cuh", os.path.join("..", "..", "include", "espm_b200.h")]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
] + os.environ.get("ESPM_NVCC_EXTRA", "").split()      # experiments: extra -D switches (part of the build digest)


def _digest():
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def needs_build():
    stamp = os.path.join(LIBDIR, "build.stamp")
    if not os.path.exists(LIBPATH) or not os.path.exists(stamp):
        return True
    with open(stamp) as fh:
        return fh.read().strip() != _digest()


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the shared library.  Returns its path."""
    if not force and not needs_build():
        return LIBPATH
    os.makedirs(OBJDIR, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 2)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [NVCC, "-shared", "-o", LIBPATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(os.path.join(LIBDIR, "build.stamp"), "w") as fh:
        fh.write(_digest())
    return LIBPATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
