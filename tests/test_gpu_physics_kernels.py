"""Per-environment material, the kernels behind it: every f32 instantiation the identity of test_gpu_physics.py does
not reach by default (coloured with a rest table; the 256-thread kernels of CLOTHB200_NT=256, in a child process since
the knob is read once per process), what the runtime reports for the PHYS kernels against the plain ones, and the
per-thread buffer of derived rows when calls alternate between streams."""
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import test_gpu_physics as TP  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F64 = torch.float32, torch.float64


def test_identity_coloured_f32_with_rest_table():
    TP.test_identity_rows_give_the_plain_bits(F32, 1, 25, True)


# the identity cases again, in a process whose kernels run 256 threads per cloth (25x25: unordered scatter; 64x64: 256
# instead of 512); an assertion fails the child
CHILD = r"""
import sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import torch
import test_gpu_physics as TP
from gym_cloth_b200 import lib as L
F32, F64 = torch.float32, torch.float64
cases = [(F32, 0, 25, False), (F32, 0, 25, True), (F32, 1, 25, False), (F32, 1, 25, True), (F32, 1, 64, False),
         (F32, 0, 16, False), (F64, 0, 25, True), (F64, 1, 25, True)]
for c in cases:
    TP.test_identity_rows_give_the_plain_bits(*c)
import ctypes as C
P = L.default_params()
t = C.c_int(0)
L.check(L.lib().clothb200_occupancy(C.byref(P), 0, None, None, C.byref(t)), "occupancy")
print("threads", t.value, "cases", len(cases))
"""


def test_identity_with_256_thread_kernels():
    env = dict(os.environ, CLOTHB200_NT="256")
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=1200)
    assert r.returncode == 0, r.stdout[-6000:]
    assert r.stdout.strip().splitlines()[-1] == "threads 256 cases 8"


def _info(P, is_f64, mode, rt, phys):
    """[ctas_per_sm, registers, local_bytes, smem_bytes], or the return code when the grid has no kernel (f64 64x64 does
    not fit one CTA's shared memory)."""
    import ctypes as C
    from gym_cloth_b200 import lib as L
    v = [C.c_int(-1) for _ in range(4)]
    rc = L.lib().clothb200_step_kernel_info(C.byref(P), is_f64, mode, rt, phys, *[C.byref(x) for x in v])
    return [x.value for x in v] if rc == 0 else rc


@pytest.mark.parametrize("W", [25, 64, 16])
def test_phys_kernels_keep_the_occupancy_of_the_plain_ones(W):
    """cudaOccupancyMaxActiveBlocksPerMultiprocessor and the registers of the kernel each entry point launches: the PHYS
    kernels run as many cloths per SM as the plain ones, on the same shared memory (the f32 25x25 128-thread kernel: 8)."""
    P = TP._params(W)
    rows = []
    for is_f64 in (0, 1):
        for mode in (0, 1):
            if mode == 1 and W not in (25, 64):
                continue
            for rt in ((0, 1) if not is_f64 else (1,)):
                plain, phys = _info(P, is_f64, mode, rt, 0), _info(P, is_f64, mode, rt, 1)
                rows.append((is_f64, mode, rt, plain, phys))
                if isinstance(plain, int) or isinstance(phys, int):
                    assert plain == phys == -4 and is_f64 and W == 64, (is_f64, mode, rt, plain, phys)   # UNSUPPORTED, both
                    continue
                assert phys[0] == plain[0] >= 1, (is_f64, mode, rt, plain, phys)
                assert phys[3] == plain[3], (is_f64, mode, rt, plain, phys)
    print(rows)
    if W == 25:
        f32_ref = _info(P, 0, 0, 0, 1)
        assert f32_ref[0] == 8 and f32_ref[1] <= 64, f32_ref


def test_rows_buffer_alternating_streams():
    """Two batches with different materials stepped by interleaved small update_n calls on two streams (the per-thread
    rows buffer is reused across them) end where each ends alone on the default stream."""
    n = 8
    m1, m2 = TP._draw(n, seed=29), TP._draw(n, seed=31)
    res = []
    for interleaved in (False, True):
        bs = []
        for m in (m1, m2):
            bc = TP._bc(TP._params(), n, F32)
            TP._load_pool(bc, n)
            TP._set_rows(bc, m)
            bs.append(bc)
        torch.cuda.synchronize()
        if interleaved:
            s = [torch.cuda.Stream(), torch.cuda.Stream()]
            for _ in range(20):
                for bc, st in zip(bs, s):
                    with torch.cuda.stream(st):
                        bc.update(3)
            torch.cuda.synchronize()
        else:
            for bc in bs:
                for _ in range(20):
                    bc.update(3)
            torch.cuda.synchronize()
        res.append([bc.pos.cpu().numpy() for bc in bs])
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a, b)
    assert not np.array_equal(res[0][0], res[0][1])
