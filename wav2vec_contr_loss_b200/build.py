"""Build libsupcon_b200.so (+ the test-only libsupcon_b200_test.so) in-tree with nvcc for sm_100a.

    python -m wav2vec_contr_loss_b200.build [--force] [--verbose]

libsupcon_b200.so is the product: a plain C-ABI shared object (include/supcon_b200.h); it links
the static CUDA runtime only, so it loads on a machine without a GPU driver
(the CPU-side tests check its exported symbols there).  libsupcon_b200_test.so is the same objects
plus the diagnostics of csrc/supcon_debug.h (tcgen05 one-tile kernels, plan introspection); only
tests/ and tools/ load it.
"""
import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsupcon_b200.so")
TEST_LIB_PATH = os.path.join(LIB_DIR, "libsupcon_b200_test.so")
TEST_ONLY_SOURCES = ("supcon_tc_debug.cu", "supcon_debug_api.cu")
STAMP = os.path.join(LIB_DIR, "libsupcon_b200.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-DSUPCON_BUILDING_DSO",
]


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest():
    h = hashlib.sha256()
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC)) + \
        [os.path.join(REPO_ROOT, "include", "supcon_b200.h"), os.path.abspath(__file__)]
    for f in files:
        with open(f, "rb") as fh:     # keyed by the path RELATIVE to the repo: the tree is copied to other roots (gpurun)
            h.update(os.path.relpath(f, REPO_ROOT).encode() + b"\0" + fh.read())
    return h.hexdigest()


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    return None


def _is_current(digest: str) -> bool:
    if not (os.path.isfile(LIB_PATH) and os.path.isfile(TEST_LIB_PATH) and os.path.isfile(STAMP)):
        return False
    with open(STAMP) as fh:
        return fh.read().strip() == digest


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile (if stale) and return the path of the shared library.  Safe to call from several processes at
    once (one rank per GPU): the build runs under an exclusive file lock and the others find it done.  A current
    build is returned without writing anything, so a read-only tree that was built before still works."""
    if not force and _is_current(_digest()):
        return LIB_PATH
    import fcntl
    os.makedirs(LIB_DIR, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force: bool, verbose: bool) -> str:
    digest = _digest()
    if not force and _is_current(digest):
        return LIB_PATH
    nvcc = nvcc_path()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libsupcon_b200.so")
    # the stamp marks a complete build: drop it before any file is rewritten, so that the unlocked check in build()
    # never hands out a library that is being relinked
    if os.path.isfile(STAMP):
        os.remove(STAMP)
    objs = []
    procs = []
    for src in _sources():
        obj = os.path.join(LIB_DIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-I", os.path.join(REPO_ROOT, "include"), "-I", CSRC, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            print(out, file=sys.stderr if p.returncode else sys.stdout, flush=True)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libsupcon_b200.so")
    test_objs = {os.path.join(LIB_DIR, f[:-3] + ".o") for f in TEST_ONLY_SOURCES}
    for out_path, members in ((LIB_PATH, [o for o in objs if o not in test_objs]), (TEST_LIB_PATH, objs)):
        link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out_path, *members,
                "-cudart", "static"]
        r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            print(r.stdout, file=sys.stderr)
            raise RuntimeError(f"link failed for {os.path.basename(out_path)}")
    with open(STAMP, "w") as fh:
        fh.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
