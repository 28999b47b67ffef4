"""Builds ``libnewton_b200.so`` in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""

from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnewton_b200.so")
# The PRODUCT library is built strict-fp: no FMA contraction + correctly rounded trig, so the kernels reproduce the
# CPU oracle bit for bit (tests/test_gpu_xpbd_parity.py).  Measured cost on B200 (round 2o): 10 % on the XPBD step kernel
# (137.7 vs 123.7 us, profiles/r2o_fp_modes.txt).  The contracted "fast" twin is selectable with NB2_FP=fast and held to the
# north-star tolerance instead of bit equality (tests/test_gpu_fast_fp.py).
LIB_FAST = os.path.join(HERE, "libnewton_b200_fast.so")
STRICT_FLAGS = ["-fmad=false", "-DNB2_STRICT_FP=1"]
SOURCES = ["nb2_api.cu", "nb2_collide.cu", "nb2_xpbd.cu", "nb2_featherstone.cu", "nb2_selection.cu", "nb2_peer.cu", "nb2_match.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "newton_b200.h")]
    return any(os.path.getmtime(p) > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into the product library and its strict-fp twin; returns the product path."""
    if not force and not needs_build() and os.path.exists(LIB_FAST):
        return LIB
    procs = []
    variants = ((LIB, ".o", STRICT_FLAGS), (LIB_FAST, ".fast.o", []))
    for _lib_path, suffix, extra in variants:
        flags = NVCC_FLAGS + extra
        if verbose:
            flags = flags + ["-Xptxas", "-v"]
        for src in SOURCES:
            obj = os.path.join(CSRC, src.replace(".cu", suffix))
            cmd = [_nvcc(), *flags, "-c", os.path.join(CSRC, src), "-o", obj]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    for lib_path, suffix, _extra in variants:
        objs = [os.path.join(CSRC, src.replace(".cu", suffix)) for src in SOURCES]
        subprocess.run([_nvcc(), "-shared", "-o", lib_path, *objs, "-lcudart"], check=True)
    return LIB


def build_variant(tag: str, defines: list[str], strict: bool = True, sources=None) -> str:
    """Builds ``libnewton_b200_<tag>.so`` from the current sources, with extra nvcc flags if any (select it with ``NB2_LIB``).

    Building it from another commit's checkout gives the baseline library that ``scripts/xpbd_lib_ab.sh`` compares against."""
    lib_path = os.path.join(HERE, f"libnewton_b200_{tag}.so")
    flags = NVCC_FLAGS + (STRICT_FLAGS if strict else []) + list(defines)
    procs, objs = [], []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", f".{tag}.o"))
        objs.append(obj)
        procs.append((src, subprocess.Popen([_nvcc(), *flags, "-c", os.path.join(CSRC, src), "-o", obj], stdout=subprocess.PIPE,
                                            stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError(f"nvcc failed on {src} ({tag})")
    subprocess.run([_nvcc(), "-shared", "-o", lib_path, *objs, "-lcudart"], check=True)
    return lib_path


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
