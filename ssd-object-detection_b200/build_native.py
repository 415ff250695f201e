"""Build libssdgeom.so for sm_100a, in-tree (so it travels to the GPU box with the snapshot).

    python ssd-object-detection_b200/build_native.py [--force]

Each translation unit is compiled separately (the matcher and geometry units with
-fmad=false; their exactness-critical arithmetic also uses non-contractible intrinsics), then
linked with the static CUDA runtime so the library carries no dependency on torch's CUDA
libraries.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "ssdgeom", "_lib")
LIB = os.path.join(OUT_DIR, "libssdgeom.so")
OBJ_DIR = os.path.join(HERE, "build")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

COMMON = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
          "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]
COMMON += os.environ.get("SSDG_EXTRA_NVCC_FLAGS", "").split()      # e.g. -DSSDG_MATCH_TIMING for phase clocks
UNITS = {
    "api.cu": [],
    "geom.cu": ["-fmad=false"],
    "match.cu": ["-fmad=false"],
    "glue.cu": ["-fmad=false"],
    "loss.cu": [],
    "detect.cu": [],
    "comm.cu": [],
    "eval.cu": ["-fmad=false"],
}


def _stamp() -> str:
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)) + ["../../include/ssdgeom.h"]:
        path = os.path.join(CSRC, name)
        if os.path.isfile(path):
            h.update(name.encode())
            with open(path, "rb") as f:
                h.update(f.read())
    h.update(repr(sorted(UNITS.items())).encode() + repr(COMMON).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, variant: str = "") -> str:
    """variant: a named side build (libssdgeom_<variant>.so, own object directory) for A/B measurements,
    selected at run time with SSDGEOM_LIB; flags come from SSDG_EXTRA_NVCC_FLAGS as usual."""
    global LIB, OBJ_DIR
    if variant:
        LIB = os.path.join(OUT_DIR, "libssdgeom_%s.so" % variant)
        OBJ_DIR = os.path.join(HERE, "build", variant)
    os.makedirs(OUT_DIR, exist_ok=True)
    os.makedirs(OBJ_DIR, exist_ok=True)
    stamp_file = LIB[:-3] + ".stamp"
    stamp = _stamp()
    if not force and os.path.isfile(LIB) and os.path.isfile(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    objs = []
    procs = []
    for unit, extra in UNITS.items():
        obj = os.path.join(OBJ_DIR, unit.replace(".cu", ".o"))
        cmd = [NVCC] + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, unit), "-o", obj]
        procs.append((unit, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for unit, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed on %s" % unit)
    link = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-o", LIB] + objs + ["-ldl"]
    subprocess.run(link, check=True)
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    _variant = sys.argv[sys.argv.index("--variant") + 1] if "--variant" in sys.argv else ""
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, variant=_variant))
