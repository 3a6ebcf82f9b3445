"""Builds libgspb200.so in-tree with nvcc for sm_100a (no JIT, no torch extension)."""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
LIB = os.path.join(OUT_DIR, "libgspb200.so")
SOURCES = ["runtime.cu", "cheby.cu", "cheby_tiled.cu", "graph.cu", "lanczos.cu", "halo.cu", "generate.cu", "staging.cu", "dist.cu", "cg.cu", "diffop.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libgspb200.so cannot be built")


def _stamp():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    files.append(os.path.join(ROOT, "include", "gspb200.h"))
    for f in files:
        with open(f, "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()


def _up_to_date():
    stamp_file = os.path.join(OUT_DIR, "stamp.txt")
    if not (os.path.exists(LIB) and os.path.exists(stamp_file)):
        return False
    with open(stamp_file) as fh:
        return fh.read().strip() == _stamp()


def build(force=False, verbose=False):
    """Build (if the sources changed) and return the path of the library.  One process at a
    time (flock on _lib/.lock: torchrun starts one process per GPU on the same tree); objects
    and the library are written under temporary names and renamed into place.  A library
    built from the current sources is returned without writing anything, so that a built
    tree can be used read-only."""
    if not force and _up_to_date():
        return LIB
    import fcntl
    os.makedirs(OUT_DIR, exist_ok=True)
    with open(os.path.join(OUT_DIR, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force, verbose):
    if not force and _up_to_date():
        return LIB
    stamp_file = os.path.join(OUT_DIR, "stamp.txt")
    stamp = _stamp()
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(OUT_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, "-O3", "-std=c++17", "-lineinfo", *ARCH, "-Xcompiler", "-fPIC",
               "-I", os.path.join(ROOT, "include"), "-I", CSRC,
               "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, p in procs:
        out = p.communicate()[0].decode()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
        if verbose and out:
            print(out)
    tmp_lib = LIB + ".tmp.%d" % os.getpid()
    subprocess.check_call([nvcc, "-shared", *ARCH, "-o", tmp_lib, *objs])
    os.replace(tmp_lib, LIB)
    with open(stamp_file + ".tmp", "w") as fh:
        fh.write(stamp)
    os.replace(stamp_file + ".tmp", stamp_file)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
