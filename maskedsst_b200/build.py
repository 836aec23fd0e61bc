"""Builds maskedsst_b200/libmsst.so (sm_100a only) from csrc/*.cu with nvcc.

    python -m maskedsst_b200.build [--force]

The library is built IN-TREE so it travels with the repo snapshot to the GPU box (it is git-ignored).
No torch headers are involved: the ABI is plain C (include/msst.h).
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libmsst.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest():
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, f), "rb") as fh:
                    h.update(f.encode()); h.update(fh.read())
    return h.hexdigest()


def _up_to_date(dig):
    stamp = os.path.join(OBJ, "digest.txt")
    if not (os.path.exists(LIB) and os.path.exists(stamp)):
        return False
    with open(stamp) as f:
        return f.read() == dig


def build(force=False, verbose=False):
    """Serialised across processes (torchrun ranks may all find the library stale): an exclusive file lock around the whole
    build, and the library is linked to a temporary name and renamed into place, so nobody ever dlopens a partial file.
    An up-to-date library is returned before the lock is taken: loading it writes nothing, so a read-only tree works."""
    if not force and _up_to_date(_digest()):
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    import fcntl
    with open(os.path.join(OBJ, "build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force, verbose):
    stamp = os.path.join(OBJ, "digest.txt")
    dig = _digest()
    if not force and _up_to_date(dig):
        return LIB
    if not os.path.exists(NVCC):
        if os.path.exists(LIB):
            return LIB   # GPU box without sources changed: use the prebuilt library
        raise RuntimeError("nvcc not found and libmsst.so is not built")

    def cc(src):
        obj = os.path.join(OBJ, src[:-3] + ".o")
        cmd = [NVCC] + FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose and r.stderr.strip():
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 4)) as ex:
        objs = list(ex.map(cc, _sources()))
    tmp = LIB + f".tmp{os.getpid()}"
    cmd = [NVCC, "-shared", "-o", tmp] + objs + ["-lcudart", "-lcuda"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB)
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
