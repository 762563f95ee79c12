"""In-tree build of libpgmuvi_b200.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m pgmuvi_b200.build [--force]

The heavy fused kernels are explicitly instantiated per (kernel kind, padded mixture count)
in csrc/inst.cu, one object file each, compiled in parallel; csrc/cabi.cu holds the C ABI.
"""
from __future__ import annotations

import hashlib
import os
import re
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libpgmuvi_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--threads", "1",
    # compressed device code: the library shrinks from 178 MB to ~30 MB (39 translation units with
    # -lineinfo); the driver inflates it when the module is loaded
    "-Xfatbin=-compress-all", "--compress-mode=size",
]
# (KIND, QT, D) instantiations, listed once in csrc/configs.h
with open(os.path.join(CSRC, "configs.h")) as _f:
    CONFIGS = [tuple(map(int, c))
               for c in re.findall(r"^PGM_CONFIG\((\d+), (\d+), (\d+)\)", _f.read(), re.M)]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _sources_digest():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for fn in sorted(os.listdir(root)):
            if fn.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, fn), "rb") as f:
                    h.update(fn.encode())
                    h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _run(cmd):
    p = subprocess.run(cmd, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + p.stdout + p.stderr)
    return p.stdout + p.stderr


def build(force=False, verbose=False, jobs=None, only=None):
    """Compile every CUDA translation unit and link the shared library.  Returns its path.

    `only` (development): recompile just the objects whose name contains one of these substrings
    (e.g. ["k0_q4_d1", "cabi"]), reuse the other objects as they are and relink; the digest stamp is
    removed so that the next plain build() recompiles everything."""
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "digest.txt")
    digest = _sources_digest()
    if only is None and not force and os.path.exists(LIB) and os.path.exists(stamp):
        with open(stamp) as f:
            if f.read().strip() == digest:
                return LIB
    nvcc = _nvcc()
    jobs_list = []
    objs = []
    o = os.path.join(OBJ, "cabi.o")
    objs.append(o)
    jobs_list.append([nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, "cabi.cu"), "-o", o])
    for (k, q, d) in CONFIGS:
        o = os.path.join(OBJ, f"inst_k{k}_q{q}_d{d}.o")
        objs.append(o)
        jobs_list.append([nvcc, *NVCC_FLAGS, f"-DPGM_INST_KIND={k}", f"-DPGM_INST_QT={q}",
                          f"-DPGM_INST_D={d}", "-c", os.path.join(CSRC, "inst.cu"), "-o", o])
    if only is not None:
        jobs_list = [j for j in jobs_list if any(t in os.path.basename(j[-1]) for t in only)]
        if os.path.exists(stamp):
            os.remove(stamp)
    if verbose:
        for j in jobs_list:
            j.insert(1, "-Xptxas=-v")
    with ThreadPoolExecutor(max_workers=jobs or os.cpu_count() or 4) as ex:
        outs = list(ex.map(_run, jobs_list))
    if verbose:
        print("\n".join(outs))
    _run([nvcc, "-shared", "-o", LIB, *objs, "-lcudart"])
    if only is None:
        with open(stamp, "w") as f:
            f.write(digest)
    return LIB


if __name__ == "__main__":
    only = [a.split("=", 1)[1].split(",") for a in sys.argv if a.startswith("--only=")]
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv, only=only[0] if only else None)
    print(path)
