"""Builds laser_b200/lib/liblaser_b200.so with nvcc for sm_100a (in-tree, no JIT cache).

One object per translation unit, compiled in parallel (the tcgen05 kernel families are the slow ones), then one link."""
import concurrent.futures
import fcntl
import hashlib
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
OBJ_DIR = os.path.join(LIB_DIR, "obj")
LIB_PATH = os.path.join(LIB_DIR, "liblaser_b200.so")
SOURCES = ["capi.cu", "tc_f16x3.cu", "tc_tf32x3.cu", "tc_tf32x1.cu", "tc_bf16.cu"]
HEADERS = ["ptx.cuh", "f16_scale.cuh", "gemm_tc.cuh", "tc_params.h", "tc_launch.h", "tc_launch_impl.cuh", "gemm_simt.cuh", "simt_epilogue.cuh", "gemm_dmma.cuh",
           "gemm_simt_kernel.inc", "split.cuh", "layers.cuh", "capi_layers.inc", "capi_multi.inc",
           "../../include/laser_b200.h"]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",   # NOT -arch=sm_100a: tcgen05 needs the 'a' PTX target
    "-lineinfo",
    "-Xcompiler", "-fPIC",
]
LINK_FLAGS = ["-shared", "-cudart", "static",       # no libcuda/libcudart link dependency: loads on CPU-only hosts
              "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-ldl"]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build liblaser_b200.so")


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _newest_header():
    return max((os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS if os.path.exists(os.path.join(CSRC, h))), default=0.0)


STAMP_PATH = LIB_PATH + ".srchash"


def _src_digest():
    """sha256 over the flags and the contents of every source the library is made of"""
    h = hashlib.sha256(repr((NVCC_FLAGS, LINK_FLAGS)).encode())
    for name in _sources() + HEADERS:
        path = os.path.join(CSRC, name)
        if os.path.exists(path):
            h.update(name.encode() + b"\0")
            with open(path, "rb") as f:
                h.update(f.read())
    return h.hexdigest()


def _stamp():
    try:
        with open(STAMP_PATH) as f:
            return f.read().strip()
    except OSError:
        return None


def _write_stamp():
    tmp = "%s.tmp%d" % (STAMP_PATH, os.getpid())
    with open(tmp, "w") as f:
        f.write(_src_digest() + "\n")
    os.replace(tmp, STAMP_PATH)


def needs_build():
    """The library is current when the digest recorded next to it matches the sources -- a copy of the tree (the snapshot
    that travels to a GPU box) keeps contents, not modification times.  A library without a digest file falls back to
    modification times."""
    if not os.path.exists(LIB_PATH):
        return True
    stamp = _stamp()
    if stamp is not None:
        return stamp != _src_digest()
    t = os.path.getmtime(LIB_PATH)
    return _newest_header() > t or any(os.path.getmtime(os.path.join(CSRC, s)) > t for s in _sources())


def build(force=False, verbose=False):
    """Compile every CUDA source into the in-tree shared library. Returns its path.

    Safe when several processes ask at once (one rank per GPU importing the package on a box whose snapshot made the
    library look stale): one of them builds under a file lock -- objects and the library are written under temporary names
    and renamed when complete -- the others wait for the lock and find the result up to date."""
    if not force and not needs_build():
        if _stamp() is None:
            try:
                _write_stamp()       # built before digests existed and current by modification time: record it
            except OSError:
                pass
        return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():     # another process built it while this one waited
                return LIB_PATH
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force, verbose):
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    nvcc = _nvcc()
    hdr_t = _newest_header()
    tag = ".tmp%d" % os.getpid()

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.splitext(src)[0] + ".o")
        path = os.path.join(CSRC, src)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(hdr_t, os.path.getmtime(path)):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj + tag]
        subprocess.check_call(cmd, env=env)
        os.replace(obj + tag, obj)
        return obj

    srcs = _sources()
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 1)) as pool:
        objs = list(pool.map(compile_one, srcs))
    subprocess.check_call([nvcc] + LINK_FLAGS + ["-o", LIB_PATH + tag] + objs, env=env)
    os.replace(LIB_PATH + tag, LIB_PATH)
    _write_stamp()
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
