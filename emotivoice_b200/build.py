"""Builds libemotivoice_b200.so in-tree with nvcc for sm_100a (no torch involved).

    python -m emotivoice_b200.build [--force]

The shared library is the product's only compute path; there is no CPU or eager
fallback.  It is git-ignored but travels to the GPU box with the snapshot.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libemotivoice_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-cudart", "static"]


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest():
    h = hashlib.sha256()
    files = sources() + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
    files.append(os.path.join(INCLUDE, "emotivoice_b200.h"))
    for f in files:
        h.update(os.path.basename(f).encode())      # names, not absolute paths: the tree is relocated on the GPU box
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def nvcc_path():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def build(force=False, verbose=True):
    """Idempotent and safe to call from several processes at once (torchrun ranks): the check-and-compile
    section runs under an exclusive file lock, so one process compiles and the others then find the stamp."""
    import fcntl
    os.makedirs(LIB_DIR, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def up_to_date(dig=None):
    """True when the in-tree library exists and was built from the current sources and flags.  Only reads, so callers that
    must not write into the tree (bench.py) can check the library without building it."""
    stamp = os.path.join(LIB_DIR, "build.stamp")
    if not (os.path.exists(LIB_PATH) and os.path.exists(stamp)):
        return False
    with open(stamp) as f:
        return f.read().strip() == (dig or _digest())


def _build_locked(force, verbose):
    stamp = os.path.join(LIB_DIR, "build.stamp")
    dig = _digest()
    if not force and up_to_date(dig):
        if verbose:
            print("emotivoice_b200.build: up to date (sources digest %s), not recompiled" % dig[:12], flush=True)
        return LIB_PATH
    objs = []
    procs = []
    for src in sources():
        obj = os.path.join(LIB_DIR, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = [nvcc_path()] + NVCC_FLAGS + ["-I", INCLUDE, "-c", src, "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out.decode())
            raise RuntimeError("nvcc failed on %s" % src)
        if verbose and out.strip():
            print(out.decode())
    cmd = [nvcc_path(), "-shared", "-o", LIB_PATH] + objs + ["-cudart", "static",
                                                           "-gencode", "arch=compute_100a,code=sm_100a"]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    with open(stamp, "w") as f:
        f.write(dig)
    if verbose:
        print("emotivoice_b200.build: compiled %d sources with nvcc for sm_100a (digest %s)" % (len(objs), dig[:12]), flush=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
