"""Build libfmb200.so (hand-written sm_100a CUDA + C-ABI) in-tree with nvcc.

The shared library is the product; there is no Python/CPU fallback.  `build()` is idempotent: it recompiles
only when a source file is newer than the library.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libfmb200.so")
SOURCES = ["fmb_lib.cu", "fmb_search.cu", "fmb_engine.cu", "fmb_build.cu", "fmb_io.cu", "fmb_extract.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libfmb200.so cannot be built")


STAMP = os.path.join(HERE, "libfmb200.stamp")
LOCK = os.path.join(HERE, ".build.lock")


def _fingerprint():
    """hash of everything the library is built from (sources, the C-ABI header, flags): file times do not survive a copy of the
    tree to another machine, contents do"""
    import hashlib
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS + os.environ.get("FMB_NVCC_EXTRA", "").split()).encode())
    paths = [os.path.join(HERE, "..", "include", "fmb200.h")]
    for root, _, files in sorted(os.walk(CSRC)):
        paths += [os.path.join(root, f) for f in sorted(files)]
    for path in paths:
        h.update(os.path.basename(path).encode())
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def needs_build():
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as f:
        return f.read().strip() != _fingerprint()


def build(force=False, verbose=False):
    """idempotent and safe when several processes call it at once (one rank per GPU under torchrun): an exclusive file lock
    serialises them, the first one builds, the others find the stamp up to date; the library is linked under a temporary name and
    renamed into place, so a process never maps a half-written file"""
    if not force and not needs_build():
        return LIB
    import fcntl
    with open(LOCK, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or needs_build():
                _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


def _build_locked(verbose):
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    extra = os.environ.get("FMB_NVCC_EXTRA", "").split()      # experiments only, e.g. -DFMB_SCHEME_MINB=4
    # one nvcc per translation unit, in parallel, then one link step
    procs = []
    for src in srcs:
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        outp, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(outp)
            raise RuntimeError(f"nvcc failed on {src}")
        if verbose:
            sys.stderr.write(outp)
        objs.append(obj)
    tmp = LIB + ".tmp.%d" % os.getpid()
    proc = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs, capture_output=True, text=True)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError("nvcc failed linking libfmb200.so")
    os.replace(tmp, LIB)
    with open(STAMP + ".tmp", "w") as f:
        f.write(_fingerprint() + "\n")
    os.replace(STAMP + ".tmp", STAMP)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
