"""Builds libmrgan.so (the C-ABI of include/mrgan.h) in-tree with nvcc for sm_100a.

Staleness is decided by a content hash of the sources and flags (side-car file ``libmrgan.so.hash``), not by mtimes, so
a snapshot copied to another box is never rebuilt needlessly and an edited source is never ignored.  Concurrent
builders (torchrun ranks on a fresh checkout) serialise on a file lock; the library appears atomically (os.replace).
"""
import fcntl
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmrgan.so")
HASH = LIB + ".hash"
LOCK = os.path.join(HERE, ".build.lock")
SOURCES = ["mrgan_api.cu"]
HEADERS = ["common.cuh", "kernels_simt.cuh", "kernels_tc.cuh", "kernels_svm.cuh", "kernels_dp.cuh", os.path.join("..", "..", "include", "mrgan.h")]
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "-shared", "-ldl", "-lcuda"]


def source_hash():
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for s in SOURCES + HEADERS:
        p = os.path.join(CSRC, s)
        if os.path.exists(p):
            with open(p, "rb") as f:
                h.update(s.encode() + b"\0" + f.read())
    return h.hexdigest()


def _stale():
    if not os.path.exists(LIB) or not os.path.exists(HASH):
        return True
    with open(HASH) as f:
        return f.read().strip() != source_hash()


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: libmrgan.so cannot be built (there is no CPU fallback)")
    return p


def build(force=False, verbose=False):
    """Compile csrc/*.cu -> mr_gan_b200/libmrgan.so if the sources changed.  Returns the library path."""
    if not force and not _stale():
        return LIB
    with open(LOCK, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():      # another process built it while we waited
                return LIB
            want = source_hash()
            fd, tmp = tempfile.mkstemp(prefix=".libmrgan.", suffix=".so.tmp", dir=HERE)
            os.close(fd)
            flags = list(FLAGS) + (["-Xptxas", "-v"] if verbose else [])
            cmd = [nvcc_path()] + flags + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", tmp]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                if os.path.exists(tmp):
                    os.unlink(tmp)
                raise RuntimeError("nvcc failed (exit %d): %s" % (r.returncode, " ".join(cmd)))
            os.replace(tmp, LIB)
            with open(HASH + ".tmp", "w") as f:
                f.write(want + "\n")
            os.replace(HASH + ".tmp", HASH)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
