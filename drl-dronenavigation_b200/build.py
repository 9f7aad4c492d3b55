"""Builds ``libdronenav.so`` (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

Each ``csrc/*.cu`` is compiled to its own object (in parallel, only when stale) and the objects are linked into the
one shared library the package loads."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ_DIR = os.path.join(PKG_DIR, "build")
LIB_PATH = os.path.join(PKG_DIR, "libdronenav.so")
INC = os.path.join(PKG_DIR, "..", "include")
# source -> headers it includes
SOURCES = {
    "dronenav.cu": ["dn_params.h", "dn_device.cuh", "dn_philox.cuh", "dn_host.h", os.path.join(INC, "dronenav.h")],
    "ppo_update.cu": ["dn_umma.cuh", "ppo_kernels.cuh", "dn_philox.cuh", "ppo_comm.cuh", "sac_kernels.cuh", os.path.join(INC, "dronenav.h"),
                      os.path.join(INC, "dnppo.h"), os.path.join(INC, "dnsac.h")],
}

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libdronenav.so cannot be built (there is no CPU fallback)")


def _obj(src: str) -> str:
    return os.path.join(OBJ_DIR, os.path.splitext(src)[0] + ".o")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _deps(src: str):
    return [os.path.join(CSRC, src)] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in SOURCES[src]] + [os.path.abspath(__file__)]


def needs_build() -> bool:
    return any(_stale(_obj(s), _deps(s)) for s in SOURCES) or _stale(LIB_PATH, [_obj(s) for s in SOURCES])


def _compile(src: str, verbose: bool) -> str:
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", _obj(src), os.path.join(CSRC, src)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return res.stdout + res.stderr


def build(force: bool = False, verbose: bool = False, only=None) -> str:
    """Compile csrc/*.cu into libdronenav.so; returns the library path."""
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    todo = [s for s in SOURCES if (force and (only is None or s in only)) or _stale(_obj(s), _deps(s))]
    with ThreadPoolExecutor(max_workers=max(1, len(todo))) as pool:
        logs = list(pool.map(lambda s: _compile(s, verbose), todo))
    cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + [_obj(s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print("\n".join(logs))
    return LIB_PATH


if __name__ == "__main__":
    import sys
    only = [a for a in sys.argv[1:] if a.endswith(".cu")] or None
    print(build(force=True, verbose=True, only=only))
