"""Builds libmapf_b200.so (the C-ABI shared library of include/mapf_b200.h) in-tree with nvcc for sm_100a.

Incremental and content-addressed: every .cu is compiled to an object under csrc/_obj/ whose sidecar records the SHA-256 of
(that source, every .cuh, the public header, the flags); the library's sidecar records the hash of all objects' keys.
Nothing depends on file times, so a prebuilt library that travelled to another box (gpurun snapshot, git checkout) is
reused exactly when its sources are the ones it was built from, and rebuilt otherwise.
"""
from __future__ import annotations

import fcntl
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB_PATH = os.path.join(_PKG, "libmapf_b200.so")
HEADER = os.path.join(os.path.dirname(_PKG), "include", "mapf_b200.h")
SOURCES = ["mapf_api.cu", "step.cu", "step_wide.cu", "observe.cu", "observe_wide.cu", "step_observe.cu",
           "step_observe_wide.cu", "bfs.cu", "gae.cu", "glue.cu", "scenario_gen.cu", "ppo_loss.cu", "obs_bits.cu",
           "astar4.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=default"]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "shared"]


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _sha(*chunks: bytes) -> str:
    h = hashlib.sha256()
    for c in chunks:
        h.update(c)
        h.update(b"\0")
    return h.hexdigest()


def _common_key() -> bytes:
    parts = [" ".join(NVCC_FLAGS).encode(), open(HEADER, "rb").read()]
    for f in sorted(os.listdir(CSRC)):
        if f.endswith(".cuh"):
            parts.append(f.encode())
            parts.append(open(os.path.join(CSRC, f), "rb").read())
    return _sha(*parts).encode()


def _object_key(src: str, common: bytes) -> str:
    return _sha(common, src.encode(), open(os.path.join(CSRC, src), "rb").read())


def _read(path: str) -> str:
    try:
        return open(path).read().strip()
    except OSError:
        return ""


def _lib_key(keys) -> str:
    return _sha(" ".join(LINK_FLAGS).encode(), *[k.encode() for k in keys])


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    common = _common_key()
    return _read(LIB_PATH + ".key") != _lib_key([_object_key(s, common) for s in _sources()])


def build(force: bool = False, verbose: bool = False) -> str:
    if not (force or _stale()):
        return LIB_PATH
    # several ranks of one job may get here at once (torchrun): one of them builds, the others wait and re-check
    with open(os.path.join(_PKG, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not (force or _stale()):
                return LIB_PATH
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force: bool, verbose: bool) -> str:
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    common = _common_key()
    srcs = _sources()
    keys = [_object_key(s, common) for s in srcs]

    def compile_one(item):
        src, key = item
        obj = os.path.join(OBJ, src[:-3] + ".o")
        if not force and os.path.exists(obj) and _read(obj + ".key") == key:
            return src, 0, ""
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj + ".tmp"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode == 0:
            os.replace(obj + ".tmp", obj)
            open(obj + ".key", "w").write(key)
        return src, r.returncode, r.stdout + r.stderr

    with ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 4)) as ex:
        results = list(ex.map(compile_one, zip(srcs, keys)))
    failed = [r for r in results if r[1] != 0]
    for src, rc, log in results:
        if log and (verbose or rc != 0):
            sys.stderr.write(f"---- {src}\n{log}")
    if failed:
        raise RuntimeError("nvcc failed building libmapf_b200.so: " + ", ".join(f[0] for f in failed))
    cmd = [nvcc] + LINK_FLAGS + [os.path.join(OBJ, s[:-3] + ".o") for s in srcs] + ["-o", LIB_PATH + ".tmp"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed linking libmapf_b200.so")
    os.replace(LIB_PATH + ".tmp", LIB_PATH)          # atomic: a concurrently loading process never sees a partial file
    open(LIB_PATH + ".key", "w").write(_lib_key(keys))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="-f" in sys.argv, verbose="-v" in sys.argv))
