"""The f32 build's reward terms and grip test keep one rounding per double operator (no DFMA), checked in its SASS.

The f32 units are compiled with FMA contraction on, and ptxas applies it to double arithmetic as well: left alone it
fuses the grip test `dx*dx + dy*dy`, the hull's turn test and shoelace sum, and the variance sum `v += d*d` into DFMAs,
and the f32 build then grips, covers and scores differently from the oracle (built with -ffp-contract=off) on the same
state.  cloth_device.cuh writes these with the __dmul_rn / __dadd_rn / __dsub_rn intrinsics, which ptxas never fuses.

For every f32 object of the build (cloth_f32.o, cloth_inst*_f32_*.o) this disassembles the SASS with line information
(build.py passes -lineinfo) and fails if a DFMA is attributed to a line inside one of those functions.  IEEE double
division (`/ N`, `0.001 / var`) is a reciprocal refined by DFMAs: those lines are exempt.  The functions' line ranges
are found in the source each time.  Skipped when the objects or the CUDA binary utilities are absent.
"""
import glob
import os
import re
import shutil
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gym_cloth_b200", "csrc")
OBJ = os.path.join(CSRC, "_build")
SOURCE = os.path.join(CSRC, "cloth_device.cuh")
# the double arithmetic the oracle comparison of coverage, variance_inv and the grip set rests on
FUNCTIONS = ("dist2_rn", "cross_rn", "grab_top", "hull_area", "block_sum", "variance_inv")


def _tool(name):
    for d in (os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH")):
        if d and os.path.exists(os.path.join(d, "bin", name)):
            return os.path.join(d, "bin", name)
    found = shutil.which(name)
    if found:
        return found
    nvcc = shutil.which(os.environ.get("NVCC", "nvcc"))
    for d in ([os.path.dirname(nvcc)] if nvcc else []) + ["/usr/local/cuda/bin"]:
        if os.path.exists(os.path.join(d, name)):
            return os.path.join(d, name)
    return None


def function_ranges(path=SOURCE):
    """{name: (first line, last line)} (1-based) of each function in FUNCTIONS: from its signature to the brace that
    closes its body."""
    lines = open(path).read().split("\n")
    out = {}
    for name in FUNCTIONS:
        sig = re.compile(r"__device__ __forceinline__ [\w:<> ]*\b%s\(" % name)
        starts = [i for i, ln in enumerate(lines) if sig.search(ln)]
        assert len(starts) == 1, (name, starts)
        i0 = starts[0]
        depth, opened = 0, False
        for i in range(i0, len(lines)):
            code = lines[i].split("//")[0]
            depth += code.count("{") - code.count("}")
            opened |= "{" in code
            if opened and depth == 0:
                out[name] = (i0 + 1, i + 1)
                break
        assert name in out, name
    return out


def division_lines(path=SOURCE):
    """Lines whose code (comments stripped) divides."""
    return {i + 1 for i, ln in enumerate(open(path).read().split("\n")) if re.search(r"[^/*]/[^/*]", ln.split("//")[0])}


def dfma_lines(obj, cuobjdump, nvdisasm):
    """{line of cloth_device.cuh: number of DFMAs attributed to it} in the SASS of one object file."""
    counts = {}
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([cuobjdump, "-xelf", "all", obj], cwd=tmp, check=True, stdout=subprocess.DEVNULL)
        cubins = glob.glob(os.path.join(tmp, "*.cubin"))
        assert cubins, obj
        for cubin in cubins:
            r = subprocess.run([nvdisasm, "--print-line-info", "-c", cubin], check=True, stdout=subprocess.PIPE, text=True)
            where = None
            for ln in r.stdout.split("\n"):
                m = re.match(r'\s*//## File "([^"]+)", line (\d+)', ln)
                if m:
                    where = int(m.group(2)) if os.path.basename(m.group(1)) == "cloth_device.cuh" else None
                elif where is not None and re.search(r"\bDFMA\b", ln):
                    counts[where] = counts.get(where, 0) + 1
    return counts


def f32_objects():
    return sorted(glob.glob(os.path.join(OBJ, "cloth_f32.o")) + glob.glob(os.path.join(OBJ, "cloth_inst*_f32_*.o")))


def contracted(obj, cuobjdump, nvdisasm, source=SOURCE):
    """[(function, line, DFMA count)] of fused double operations inside FUNCTIONS, division lines excepted."""
    ranges, div = function_ranges(source), division_lines(source)
    bad = []
    for line, n in sorted(dfma_lines(obj, cuobjdump, nvdisasm).items()):
        for name, (a, b) in ranges.items():
            if a <= line <= b and line not in div:
                bad.append((name, line, n))
    return bad


def test_function_ranges_are_found():
    r = function_ranges()
    assert set(r) == set(FUNCTIONS)
    for name, (a, b) in r.items():
        assert a <= b, name
    assert r["grab_top"][1] - r["grab_top"][0] > 20 and r["hull_area"][1] - r["hull_area"][0] > 30


@pytest.mark.parametrize("obj", [os.path.basename(o) for o in f32_objects()] or ["(not built)"])
def test_f32_reward_terms_and_grip_test_are_not_contracted(obj):
    if obj == "(not built)":
        pytest.skip("no f32 objects in %s: run `python -m gym_cloth_b200.build`" % OBJ)
    cuobjdump, nvdisasm = _tool("cuobjdump"), _tool("nvdisasm")
    if not cuobjdump or not nvdisasm:
        pytest.skip("cuobjdump / nvdisasm not found")
    path = os.path.join(OBJ, obj)
    if os.path.getmtime(path) < os.path.getmtime(SOURCE):
        pytest.skip("%s is older than cloth_device.cuh: rebuild first" % obj)
    bad = contracted(path, cuobjdump, nvdisasm)
    assert not bad, "DFMA inside (function, line of cloth_device.cuh, count): %s" % bad
