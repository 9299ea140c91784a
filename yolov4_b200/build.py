"""Compiles csrc/*.cu into yolov4_b200/libyolohead.so for sm_100a (nvcc cross-compiles without a GPU).

The .so is built in-tree (git-ignored, but it travels to the GPU box with the repo snapshot).
"""
import fcntl
import glob
import hashlib
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libyolohead.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",                      # no FMA contraction: the reference rounds a*b and +c separately
    "-Xcompiler", "-fPIC",
]


def _nvcc():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found; libyolohead.so cannot be built")
    return p


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _deps():
    return sources() + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + sorted(glob.glob(os.path.join(HERE, "..", "include", "*.h")))


def source_hash():
    """Hash of everything the library is compiled from; embedded in the .so (yl_source_hash()) and in a side file, so that
    a library built from other sources is never loaded silently (file times do not survive a snapshot copy)."""
    h = hashlib.sha256()
    for d in _deps():
        h.update(os.path.basename(d).encode())
        h.update(open(d, "rb").read())
    return h.hexdigest()[:16]


def is_stale():
    if not os.path.exists(LIB) or not os.path.exists(LIB + ".srchash"):
        return True
    return open(LIB + ".srchash").read().strip() != source_hash()


def build_lib(force=False, verbose=False, extra=(), out=None, only=None):
    """extra: additional nvcc flags (e.g. -DYL_FT_STAGES=4 for tuning builds); out: alternative output path;
    only: basenames of the sources the extra flags apply to (the other objects are those of the default build)."""
    if out is None and not force and not is_stale():
        return LIB
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    with open(os.path.join(bdir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)                 # ranks of one job build once, not concurrently into one file
        try:
            if out is None and not force and not is_stale():
                return LIB
            return _build_locked(bdir, verbose, extra, out, only)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(bdir, verbose, extra, out, only):
    objs = []
    procs = []
    sh = source_hash()
    for src in sources():
        obj = os.path.join(bdir, os.path.basename(src)[:-3] + ".o")
        variant = out is not None and (only is None or os.path.basename(src) in only)
        if out is not None and not variant:
            if not os.path.exists(obj):
                raise RuntimeError("build the default library first (%s is missing)" % obj)
            objs.append(obj)
            continue
        if variant:
            obj = obj[:-2] + "." + os.path.basename(out) + ".o"
        cmd = [_nvcc()] + NVCC_FLAGS + ['-DYL_SOURCE_HASH="%s"' % sh] + (list(extra) if (variant or out is None) else []) + \
              (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, p in procs:
        log, _ = p.communicate()
        if verbose and log:
            print(log)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s" % (" ".join(cmd), log))
    target = out or LIB
    cmd = [_nvcc(), "-shared", "-o", target + ".tmp"] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(cmd)
    os.replace(target + ".tmp", target)
    if out is None:
        with open(LIB + ".srchash", "w") as f:
            f.write(sh + "\n")
    return target


if __name__ == "__main__":
    import sys
    print(build_lib(force=True, verbose="-v" in sys.argv))
