"""In-tree build of librover_b200.so (explicit nvcc, sm_100a only; no JIT cache)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librover_b200.so")
SOURCES = ["terrain.cu", "raycast.cu", "raycast_tiled.cu", "raycast_shadow.cu", "rock.cu", "task.cu", "step.cu", "stones.cu", "knn.cu", "policy.cu", "hooks.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false",                 # bit-exact parity: never contract mul+add
              "--threads", "0",              # one compilation per source file in parallel (74 s -> 12 s); same object code
              "-Xcompiler", "-fPIC", "-shared",
              "-Xlinker", "--no-undefined"]   # a declaration that no source defines fails the link, not the library's load


def _nvcc():
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


HASH_FILE = LIB + ".srchash"
LOCK_FILE = LIB + ".lock"


def source_hash():
    """sha256 over the sources, the public header and the compiler flags (mtimes do not survive a copy of the tree)."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh")))
    files.append(os.path.join(HERE, "..", "include", "rover_b200.h"))
    for f in files:
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def raycast_hash():
    """sha256 over the sources of the heightmap ray-cast kernels alone: what profiles/raycast_traffic.json (an ncu capture of
    that kernel) is tied to -- bench.py quotes the capture only for the build it was taken from."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for f in ("common.cuh", "raycast_common.cuh", "shadow_bounds.cuh", "raycast_shadow.cu", "raycast_tiled.cu"):
        h.update(f.encode())
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def needs_build():
    if not os.path.exists(LIB):
        return True
    try:
        with open(HASH_FILE) as fh:
            return fh.read().strip() != source_hash()
    except OSError:
        return True


def build(force=False, verbose=False):
    """Compile under an exclusive file lock into a temporary file and rename it into place: the ranks of a multi-GPU
    launch never see a half-written library, and only one of them compiles."""
    import fcntl
    if not force and not needs_build():
        return LIB
    with open(LOCK_FILE, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():          # another process built it while we waited
                return LIB
            tmp = LIB + ".tmp.%d" % os.getpid()
            cmd = [_nvcc()] + NVCC_FLAGS + ["-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
            if verbose:
                print(r.stderr)
            os.replace(tmp, LIB)
            with open(HASH_FILE + ".tmp", "w") as fh:
                fh.write(source_hash())
            os.replace(HASH_FILE + ".tmp", HASH_FILE)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB
