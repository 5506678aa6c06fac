#!/usr/bin/env python
"""Build gym_cloth_b200/libclothb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m gym_cloth_b200.build [--force] [--verbose]

Translation units, compiled in parallel: cloth_f32.cu (production entry points + renderer), cloth_f64.cu (parity
build, -fmad=false so that every operator is one rounded IEEE operation), cloth_abi.cu (extern "C" surface) and
cloth_inst.cu twelve times (the step kernel per scalar type, compile-time grid width, and batch or per-environment
material).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libclothb200.so")
OBJ = os.path.join(HERE, "csrc", "_build")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
# f32 (production): flush-to-zero and approximate div/sqrt - the parity contract of this build is a tolerance, and
# IEEE fix-up sequences around every rsqrt/division are pure latency on the serial replay paths.
# f64 (parity): no FMA contraction, IEEE everything.
F32 = ["-ftz=true", "-prec-div=false", "-prec-sqrt=false"]
F64 = ["-fmad=false"]
# (source, object name, flags); cloth_inst.cu holds the step kernel for one (scalar type, grid width) pair, with the
# batch's material or (cloth_inst_phys_*) with per-environment material rows
UNITS = [("cloth_f32.cu", "cloth_f32.o", F32), ("cloth_f64.cu", "cloth_f64.o", F64), ("cloth_abi.cu", "cloth_abi.o", [])]
for _t, _sfx, _fl in (("float", "f32", F32), ("double", "f64", F64)):
    for _w in (25, 0, 64):
        UNITS.append(("cloth_inst.cu", "cloth_inst_%s_w%d.o" % (_sfx, _w), _fl + ["-DCLOTH_T=%s" % _t, "-DCLOTH_INSTANTIATE_WC=%d" % _w]))
        UNITS.append(("cloth_inst.cu", "cloth_inst_phys_%s_w%d.o" % (_sfx, _w),
                      _fl + ["-DCLOTH_T=%s" % _t, "-DCLOTH_INSTANTIATE_WC=%d" % _w, "-DCLOTH_INSTANTIATE_PHYS=1"]))


def _newest_src():
    t = 0
    for root, _, files in os.walk(CSRC):
        if "_build" in root:
            continue
        for f in files:
            if f.endswith((".cu", ".cuh", ".h")):
                t = max(t, os.path.getmtime(os.path.join(root, f)))
    t = max(t, os.path.getmtime(os.path.join(HERE, "..", "include", "clothb200.h")))
    return t


LIB_IEEE = os.path.join(HERE, "libclothb200_f32ieee.so")
# study variant of the f32 build: the reference's expressions in float (sqrt and division as written, no rsqrt forms),
# IEEE-rounded div/sqrt, denormals kept, FMA contraction as in production.  Only the f32 entry points are meaningful.
IEEE = ["-DCLOTHB200_F32_REFERENCE_FORMS", "-ftz=false", "-prec-div=true", "-prec-sqrt=true"]
UNITS_IEEE = [("cloth_f32.cu", "ieee_cloth_f32.o", IEEE), ("cloth_f64.cu", "cloth_f64.o", None), ("cloth_abi.cu", "cloth_abi.o", None)]
for _w in (25, 0, 64):
    UNITS_IEEE.append(("cloth_inst.cu", "ieee_cloth_inst_f32_w%d.o" % _w, IEEE + ["-DCLOTH_T=float", "-DCLOTH_INSTANTIATE_WC=%d" % _w]))
    UNITS_IEEE.append(("cloth_inst.cu", "ieee_cloth_inst_phys_f32_w%d.o" % _w,
                       IEEE + ["-DCLOTH_T=float", "-DCLOTH_INSTANTIATE_WC=%d" % _w, "-DCLOTH_INSTANTIATE_PHYS=1"]))
    UNITS_IEEE.append(("cloth_inst.cu", "cloth_inst_f64_w%d.o" % _w, None))
    UNITS_IEEE.append(("cloth_inst.cu", "cloth_inst_phys_f64_w%d.o" % _w, None))


def build_ieee(force=False, verbose=False):
    """libclothb200_f32ieee.so (needs the objects of the main build for the shared f64 / ABI units)."""
    build(force=False, verbose=verbose)
    if not force and os.path.exists(LIB_IEEE) and os.path.getmtime(LIB_IEEE) >= _newest_src():
        return LIB_IEEE
    return _build(LIB_IEEE, [u for u in UNITS_IEEE], verbose)


def build(force=False, verbose=False):
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_src():
        return LIB
    return _build(LIB, UNITS, verbose)


def _build(LIB, UNITS, verbose):
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ, exist_ok=True)
    procs = []
    objs = []
    for src, oname, extra in UNITS:
        obj = os.path.join(OBJ, oname)
        if extra is None:            # reuse the object of the main build
            objs.append(obj)
            continue
        objs.append(obj)
        cmd = [nvcc] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            print(" ".join(cmd)); print(out)
        if p.returncode:
            raise RuntimeError("nvcc failed for %s" % cmd[-3])
    cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
    if "--ieee" in sys.argv:
        print(build_ieee(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
