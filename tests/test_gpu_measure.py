"""What the agent sees, held to the oracle bit for bit in both builds: coverage, variance_inv, the out-of-bounds flag,
the reward / done bookkeeping and the grip set.

All of these run in double in both builds (cloth_device.cuh: grab_top, hull_area, variance_inv, out_of_bounds; the
bookkeeping at the end of cloth_step_kernel).  The f32 build widens each stored coordinate to double, so on the same
state it must give the same bits as the f64 build and the oracle (oracle/cloth_oracle.c, -ffp-contract=off) - with
one documented exception: the f32 units widen under flush-to-zero, so a subnormal stored coordinate reads as a zero
of its sign (DESIGN.md section 4; the physics never makes one, only set_state can).

1. clothb200_measure_{f32,f64} over families of constructed states (a monotone chain's hard cases: piles of clipped
   duplicates on the square's edges, collinear and one-point sets, ties in x, points in convex position, N not a
   power of two), per width: coverage == oracle hull_area (and scipy's ConvexHull to 1e-12), variance_inv == a numpy
   restatement of the kernel's summation order (and math.fsum to 1e-13), the OOB flag == the oracle's at the exact
   thresholds; env_order subsets, NaN rows, subnormal coordinates.
2. The same rows at the end of a step whose grip catches nothing, through every step-kernel family.
3. After real f32 actions (25x25, and 64x64 coloured as bench.py config 4), the returned state's measurement.
4. The bookkeeping at its boundaries (coverage exactly 0.92, the last action, reward types, initialize).
5. The grip radius test on its boundary: points a few ulps inside / outside, where a fused multiply-add would decide
   differently from the oracle's rounded expression; grab_top alone, at the start of a step and under force_grab.
"""
import ctypes as C
import json
import math
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

from conftest import load_golden

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle.oracle import OracleCloth  # noqa: E402  (checker only)
from test_gpu_widths import _oparams, _params  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64, F32 = torch.float64, torch.float32
W_F64 = [3, 4, 8, 11, 12, 16, 24, 25, 26, 32, 33, 40, 55]
W_F32 = W_F64 + [56, 64, 65, 75]     # 55 and 75: the largest grids one CTA holds in f64 / f32
CASES = [("f64", W) for W in W_F64] + [("f32", W) for W in W_F32]
DT = {"f64": F64, "f32": F32}
NP = {"f64": np.float64, "f32": np.float32}


def _L():
    from gym_cloth_b200 import lib as L
    return L


def _bc(P, n, dt, mode=None):
    from gym_cloth_b200.batched import BatchedCloth
    L = _L()
    return BatchedCloth(P, n, dtype=DT[dt], mode=L.MODE_REFERENCE_ORDER if mode is None else mode)


def _nt(W):
    """Threads per cloth of the kernel a W x W grid runs on (cloth_abi.cu threads_per_cloth, launch_step_nt)."""
    nt = int(os.environ.get("CLOTHB200_NT", "0") or 0)
    if nt not in (128, 256, 512):
        nt = 512 if W >= 64 else 128
    if W != 64 and nt == 512:
        return 128
    return nt


def _stored(a, dt):
    """The values a state holds once stored in dtype dt, as doubles (f32: round to nearest, then widen exactly)."""
    return np.asarray(a, np.float64).astype(NP[dt]).astype(np.float64)


def _flush(a, dt):
    """What the kernels read: in f32 a subnormal stored value reads as a zero of its sign (see the module docstring)."""
    a = np.array(a, np.float64)
    if dt == "f32":
        sub = (a != 0) & (np.abs(a) < np.finfo(np.float32).tiny)
        a[sub] = np.copysign(0.0, a[sub])
    return a


# ---------------------------------------------------------------------------------------------- references
def _block_sum(per_thread, NT):
    """ClothCTA::block_sum: xor butterfly 16, 8, 4, 2, 1 in each warp, then a sequential sum over warps from 0.0."""
    v = np.asarray(per_thread, np.float64).reshape(NT // 32, 32)
    lane = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = v + v[:, lane ^ o]
    s = 0.0
    for w in range(NT // 32):
        s = s + v[w, 0]
    return s


def _strided(x, NT):
    """Per-thread sums over p = tid, tid+NT, ... from 0.0 (padding adds +0.0, which changes no such sum)."""
    cols = -(-len(x) // NT)
    a = np.zeros(cols * NT)
    a[:len(x)] = x
    a = a.reshape(cols, NT)
    s = np.zeros(NT)
    for c in range(cols):
        s = s + a[c]
    return s


def variance_inv_kernel_order(z, NT):
    """ClothCTA::variance_inv restated: every operator one IEEE double rounding, in the kernel's order."""
    z = np.asarray(z, np.float64)
    N = len(z)
    mean = _block_sum(_strided(z, NT), NT) / N
    d = z - mean
    var = _block_sum(_strided(d * d, NT), NT) / N
    return 1000.0 if var < 0.000001 else 0.001 / var, var


def variance_inv_fsum(z):
    z = [float(v) for v in z]
    mean = math.fsum(z) / len(z)
    var = math.fsum((v - mean) ** 2 for v in z) / len(z)
    return 1000.0 if var < 0.000001 else 0.001 / var, var


def _scipy_area(xy):
    from scipy.spatial import ConvexHull
    from scipy.spatial import QhullError
    try:
        return ConvexHull(np.unique(xy, axis=0)).volume
    except (QhullError, ValueError):
        return 0.0       # the reference's QhullError branch (cloth_env.py:634-637)


def _oracle(W, pos):
    """(coverage, out_of_bounds) of the oracle on a [N, 3] double state."""
    o = OracleCloth(_oparams(W))
    o.set_state(pos, pos, np.zeros(len(pos), np.uint8))
    return o.coverage(), o.out_of_bounds()


# ---------------------------------------------------------------------------------------------- state families
def _grid(W):
    r, c = np.meshgrid(np.arange(W), np.arange(W), indexing="ij")
    return np.stack([r / (W - 1.0), c / (W - 1.0), np.zeros((W, W))], -1).reshape(-1, 3)


def families(W, dt):
    """[(name, [N, 3] doubles)] - each already a value of dtype dt."""
    N = W * W
    rng = np.random.RandomState(1000 + W)
    z = lambda: rng.uniform(0.0, 0.2, N)
    g = _grid(W)
    out = [("flat", g.copy())]
    s = g.copy(); s[:, 0] += 0.3; s[:, 1] -= 0.2; s[:, 2] = z(); out.append(("shifted", s))
    s = g.copy(); s[:, :2] = (s[:, :2] - 0.5) * 3 + 0.5; s[:, 2] = z(); out.append(("scaled3", s))
    s = np.stack([rng.uniform(1.01, 1.2, N), rng.uniform(-0.2, 1.2, N), z()], -1); out.append(("right_of_square", s))
    s = np.stack([rng.uniform(-0.2, -0.01, N), rng.uniform(-0.2, -0.01, N), z()], -1); out.append(("below_left", s))
    t = rng.uniform(0, 1, N)
    s = np.stack([t, 0.1 + 0.7 * t, z()], -1); out.append(("diagonal", s))
    th = 2 * np.pi * np.arange(N) / N
    s = np.stack([0.5 + 0.45 * np.cos(th), 0.5 + 0.45 * np.sin(th), z()], -1)[rng.permutation(N)]; out.append(("circle", s))
    s = np.stack([rng.uniform(-0.3, 1.3, N), rng.uniform(-0.3, 1.3, N), z()], -1); out.append(("uniform_wide", s))
    s = np.stack([rng.uniform(0, 1, N), rng.uniform(0, 1, N), z()], -1); out.append(("uniform_unit", s))
    s = g.copy(); s[:, 1] = rng.uniform(0, 1, N); s[:, 2] = z(); out.append(("columns", s))
    s = np.tile([0.2, 0.25, 0.05], (N, 1)); s[1] = [0.8, 0.25, 0.05]; s[2] = [0.5, 0.25 + 1e-12, 0.05]
    s[:, 2] += rng.uniform(0, 1e-3, N); out.append(("sliver", s))
    vals = np.array([0.0, -0.0, 1.0, 0.5])
    s = np.stack([vals[rng.randint(0, 4, N)], vals[rng.randint(0, 4, N)], z()], -1); out.append(("zeros_ones", s))
    if W == 25:
        pool = load_golden("bench_pool_t1.npz")
        out += [("pool%d" % k, pool["pos"][k]) for k in range(0, 64, 9)]
    # variance_inv on both sides of its clamp (var < 1e-6 -> 1000): z = +-a on alternate points, a tuned in dt's ulps
    below, above = _clamp_pair(W, dt)
    out += [("var_below", below), ("var_above", above)]
    return [(n, _stored(p, dt)) for n, p in out]


def _clamp_pair(W, dt):
    N = W * W
    sign = np.where(np.arange(N) % 2 == 0, 1.0, -1.0)
    sign[N - 1] = 0.0 if N % 2 else sign[N - 1]
    base = _grid(W)
    a = NP[dt](math.sqrt(1e-6 / np.mean(sign * sign)))
    step = lambda v, d: np.nextafter(v, NP[dt](d))
    for _ in range(64):                               # walk down until the kernel order's variance is below 1e-6
        zb = _stored(sign * np.float64(a), dt)
        if variance_inv_kernel_order(zb, _nt(W))[1] < 1e-6:
            break
        a = step(a, 0)
    for _ in range(64):                               # then up to the first value at or above it
        b = step(a, 1)
        zb = _stored(sign * np.float64(b), dt)
        if variance_inv_kernel_order(zb, _nt(W))[1] >= 1e-6:
            break
        a = b
    lo, hi = base.copy(), base.copy()
    lo[:, 2] = sign * np.float64(a); hi[:, 2] = sign * np.float64(b)
    assert variance_inv_kernel_order(_stored(lo[:, 2], dt), _nt(W))[1] < 1e-6 <= variance_inv_kernel_order(_stored(hi[:, 2], dt), _nt(W))[1]
    return lo, hi


def oob_rows(W, dt):
    """A flat grid with one coordinate of one point on or next to an OOB threshold (x, y >= 1.25 or < -0.25, z >= 1
    or < 0; in f32 the neighbours are f32 values)."""
    f = NP[dt]
    out = []
    for axis, vals in ((0, (1.25, np.nextafter(f(1.25), f(0)), -0.25, np.nextafter(f(-0.25), f(-1)))),
                       (1, (1.25, np.nextafter(f(1.25), f(0)), -0.25, np.nextafter(f(-0.25), f(-1)))),
                       (2, (1.0, np.nextafter(f(1.0), f(0)), -0.0, np.nextafter(f(0), f(-1))))):
        for v in vals:
            s = _grid(W)
            s[:, 2] = 0.05
            s[(W * W) // 3, axis] = float(v)
            out.append(("oob_%d_%r" % (axis, float(v)), _stored(s, dt)))
    return out


# ---------------------------------------------------------------------------------------------- measuring
def _load(bc, states):
    for e, (_, s) in enumerate(states):
        bc.set_state(s, s, None, env=e)


def _stored_back(bc, e):
    """The state as stored on the device, widened to double on the host."""
    return bc.pos[e, :, :3].cpu().numpy().astype(np.float64)


def _fresh_outputs(bc):
    bc.coverage.fill_(-7.0); bc.variance_inv.fill_(-7.0); bc.flags.fill_(-1)


def _measure(W, dt, states):
    """coverage, variance_inv, OOB flag per state through clothb200_measure_<dt> in one batch."""
    P, _ = _params(W)
    bc = _bc(P, len(states), dt)
    _load(bc, states)
    _fresh_outputs(bc)
    bc.measure()
    torch.cuda.synchronize()
    for e, (name, s) in enumerate(states):
        assert np.array_equal(_stored_back(bc, e), s), (W, dt, name)        # the state is what the expectations use
    return (bc.coverage.cpu().numpy().copy(), bc.variance_inv.cpu().numpy().copy(),
            (bc.flags.cpu().numpy() & _L().FLAG_OOB) != 0, bc)


def _expected(W, dt, states, NT=None):
    NT = _nt(W) if NT is None else NT
    cov, vinv, oob = [], [], []
    for name, s in states:
        seen = _flush(s, dt)
        c, o = _oracle(W, seen)
        cov.append(c); oob.append(o)
        vinv.append(variance_inv_kernel_order(seen[:, 2], NT)[0])
    return np.array(cov), np.array(vinv), np.array(oob)


def _bits_equal(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.int64), np.asarray(b, np.float64).view(np.int64))


def _check_rows(W, dt, states, got, exp, what):
    cov, vinv, oob = got
    ecov, evinv, eoob = exp
    bad = [(states[e][0], cov[e], ecov[e], vinv[e], evinv[e], bool(oob[e]), bool(eoob[e])) for e in range(len(states))
           if not (cov[e] == ecov[e] and _bits_equal(vinv[e], evinv[e]) and oob[e] == eoob[e])]
    assert not bad, (what, dt, W, "(row, coverage, oracle, variance_inv, restated, oob, oracle)", bad)


_MEASURED = {}


def _measured(dt, W):
    if (dt, W) not in _MEASURED:
        states = families(W, dt) + oob_rows(W, dt)
        _MEASURED[(dt, W)] = (states, _measure(W, dt, states)[:3])
    return _MEASURED[(dt, W)]


@pytest.mark.parametrize("dt,W", CASES)
def test_measure_equals_oracle_bit_for_bit(dt, W):
    states, got = _measured(dt, W)
    _check_rows(W, dt, states, got, _expected(W, dt, states), "measure")


@pytest.mark.parametrize("dt,W", CASES)
def test_measure_against_independent_references(dt, W):
    """scipy's Qhull area to 1e-12 and an fsum variance to 1e-13 relative (away from the clamp threshold)."""
    states, (cov, vinv, _) = _measured(dt, W)
    for e, (name, s) in enumerate(states):
        xy = np.clip(s[:, :2], 0.0, 1.0)
        assert abs(cov[e] - _scipy_area(xy)) <= 1e-12, (name, cov[e], _scipy_area(xy))
        ref, var = variance_inv_fsum(s[:, 2])
        if abs(var - 1e-6) > 1e-9:
            assert abs(vinv[e] - ref) <= 1e-13 * ref, (name, vinv[e], ref)
    names = [n for n, _ in states]
    e_flat, e_scaled = names.index("flat"), names.index("scaled3")
    assert cov[e_flat] == 1.0 and cov[e_scaled] == 1.0
    for n in ("right_of_square", "below_left"):
        assert cov[names.index(n)] == 0.0, n
    lo, hi = vinv[names.index("var_below")], vinv[names.index("var_above")]
    assert lo == 1000.0 and abs(hi - 1000.0) < 1e-3, (lo, hi)      # the clamp, and 0.001 / var an f32 ulp of z above it


def test_measure_nt256_child(tmp_path):
    """The variance order follows the thread count: CLOTHB200_NT=256 in a child process (read once per process)
    equals the restatement for 256 threads, and coverage and flags stay the same bits."""
    out = tmp_path / "nt256.json"
    code = ("import sys; sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + '/tests')\n"
            "import json, test_gpu_measure as T\n"
            "res = {}\n"
            "for dt, W in (('f64', 25), ('f64', 33), ('f32', 25), ('f32', 64), ('f32', 75)):\n"
            "    states, got = T._measured(dt, W)\n"
            "    T._check_rows(W, dt, states, got, T._expected(W, dt, states, NT=256), 'NT=256')\n"
            "    res['%s_%d' % (dt, W)] = [g.tolist() for g in got]\n"
            "json.dump(res, open(sys.argv[2], 'w'))\n")
    env = dict(os.environ, CLOTHB200_NT="256")
    r = subprocess.run([sys.executable, "-c", code, ROOT, str(out)], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-6000:]
    res = json.loads(out.read_text())
    for key, (cov, vinv, oob) in res.items():
        dt, W = key.split("_")[0], int(key.split("_")[1])
        _, (c0, _, o0) = _measured(dt, W)
        assert np.array_equal(np.array(cov), c0) and np.array_equal(np.array(oob), o0), key


def test_subset_writes_only_its_rows():
    """measure with an env_order subset (BatchedClothEnv._measure_subset) writes exactly the selected rows."""
    for dt in ("f32", "f64"):
        W = 25
        states = families(W, dt)
        P, _ = _params(W)
        bc = _bc(P, len(states), dt)
        _load(bc, states)
        bc.measure(); torch.cuda.synchronize()
        full = [t.clone() for t in (bc.coverage, bc.variance_inv, bc.flags, bc.obs)]
        for t, v in zip((bc.coverage, bc.variance_inv, bc.flags, bc.obs), (-3.5, -4.5, 64, -5.5)):
            t.fill_(v)
        before = [t.clone() for t in (bc.coverage, bc.variance_inv, bc.flags, bc.obs)]
        sel = [len(states) - 1, 3, 0, 7]
        bc.env_order, bc.n_env = torch.tensor(sel, dtype=torch.int32, device="cuda"), len(sel)
        try:
            bc.measure()
        finally:
            bc.env_order, bc.n_env = None, len(states)
        torch.cuda.synchronize()
        mask = torch.zeros(len(states), dtype=torch.bool, device="cuda"); mask[sel] = True
        for t, f, b in zip((bc.coverage, bc.variance_inv, bc.flags, bc.obs), full, before):
            assert torch.equal(t[mask], f[mask]), dt
            assert np.array_equal(t[~mask].cpu().numpy().view(np.uint8), b[~mask].cpu().numpy().view(np.uint8)), dt


def test_nan_row_leaves_the_others_exact():
    """A NaN coordinate in one cloth: every other row is exact, and two calls give the same bytes (the NaN row's own
    values are unspecified: the reference would raise)."""
    for dt, W in (("f64", 16), ("f32", 25), ("f32", 64)):
        states = families(W, dt)[:6]
        s = states[2][1].copy(); s[5, 0] = np.nan
        states.append(("nan_x", s))
        s = states[0][1].copy(); s[W, 2] = np.nan
        states.append(("nan_z", s))
        P, _ = _params(W)
        bc = _bc(P, len(states), dt)
        _load(bc, states)
        got = []
        for _ in range(2):
            _fresh_outputs(bc)
            bc.measure(); torch.cuda.synchronize()
            got.append([t.cpu().numpy().copy() for t in (bc.coverage, bc.variance_inv, bc.flags)])
        for a, b in zip(*got):
            assert a.tobytes() == b.tobytes(), (dt, W)
        k = len(states) - 2
        exp = _expected(W, dt, states[:k])
        _check_rows(W, dt, states[:k], (got[0][0][:k], got[0][1][:k], (got[0][2][:k] & _L().FLAG_OOB) != 0), exp, "nan")


def test_f32_subnormal_coordinates_read_as_signed_zero():
    """DESIGN.md section 4: the f32 build widens under flush-to-zero, so measure sees a subnormal stored coordinate as
    a zero of its sign.  Pinned both ways: the result equals the oracle on the flushed state, and the rows are built so
    that the unflushed state measures differently (a negative subnormal z is out of bounds for the oracle)."""
    W, dt = 25, "f32"
    tiny = float(np.finfo(np.float32).smallest_subnormal)
    g = _grid(W); g[:, 2] = 0.05
    rows = []
    s = g.copy(); s[100, 2] = -tiny; rows.append(("z_neg_subnormal", s))
    s = g.copy(); s[100, 2] = -3 * tiny; s[200, 0] = 5 * tiny; rows.append(("mixed", s))
    s = g.copy(); s[:, 0] = np.where(g[:, 0] == 0.0, -tiny, g[:, 0]); rows.append(("x_edge", s))
    s = np.tile([0.5, 0.5, 0.0], (W * W, 1)); s[::2, 0] = tiny * np.arange(1, W * W + 1, 2); s[:, 2] = 0.01
    s[1::7, 1] = 2 * tiny; rows.append(("subnormal_pile", s))
    states = [(n, _stored(p, dt)) for n, p in rows]
    assert all(np.any((p != 0) & (np.abs(p) < np.finfo(np.float32).tiny)) for _, p in states)
    got = _measure(W, dt, states)[:3]
    _check_rows(W, dt, states, got, _expected(W, dt, states), "subnormal (flushed)")
    raw = [_oracle(W, s)[1] for _, s in states]
    assert raw[0] and not got[2][0]          # the unflushed oracle would flag it: the documented difference


# ---------------------------------------------------------------------------------------------- 2. end of a step
def _plans(n, gx=-5.0, gy=-5.0, iters_pull=0):
    plans = (_L().Plan * n)()
    for p in plans:
        p.gx, p.gy, p.dxr, p.dyr, p.iters_pull = gx, gy, 0.0, 0.0, iters_pull
    return plans


STEP_FAMILIES = [("f32", 25, "ref", False), ("f64", 25, "ref", False), ("f32", 25, "col", False), ("f64", 25, "col", False),
                 ("f32", 25, "ref", True), ("f64", 25, "ref", True), ("f32", 25, "col", True), ("f32", 64, "col", False),
                 ("f32", 64, "ref", False), ("f32", 33, "ref", False), ("f64", 33, "ref", True), ("f32", 75, "ref", False)]


@pytest.mark.parametrize("dt,W,mode,phys", STEP_FAMILIES)
def test_nothing_gripped_step_measures_as_measure(dt, W, mode, phys):
    """A step whose grip catches nothing (NOGRAB, no substep) reports measure's coverage, variance_inv and flags."""
    L = _L()
    states, (mcov, mvinv, moob) = _measured(dt, W)
    P, _ = _params(W)
    bc = _bc(P, len(states), dt, L.MODE_COLOURED if mode == "col" else L.MODE_REFERENCE_ORDER)
    if phys:
        bc.set_physics()                      # the batch's own material through the _phys entry points
    _load(bc, states)
    _fresh_outputs(bc)
    bc.step_plans(_plans(len(states)))
    torch.cuda.synchronize()
    f = bc.flags.cpu().numpy()
    assert (bc.sim_steps.cpu().numpy() == 0).all() and ((f & L.FLAG_NOGRAB) != 0).all()
    assert np.array_equal(bc.coverage.cpu().numpy(), mcov)
    assert _bits_equal(bc.variance_inv.cpu().numpy(), mvinv)
    assert np.array_equal((f & L.FLAG_OOB) != 0, moob)
    for e, (name, s) in enumerate(states):
        assert np.array_equal(_stored_back(bc, e), s), name


@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_nothing_gripped_time_sliced_step_measures_as_measure(dt):
    """The same through a time-sliced launch: four resident slots for the whole batch."""
    L = _L()
    W = 25
    states, (mcov, mvinv, moob) = _measured(dt, W)
    P, _ = _params(W)
    bc = _bc(P, len(states), dt)
    _load(bc, states)
    _fresh_outputs(bc)
    L.check(L.lib().clothb200_debug_set_slicing(4, 8), "debug_set_slicing")
    try:
        n0 = L.lib().clothb200_launch_count()
        bc.step_plans(_plans(len(states)))
        torch.cuda.synchronize()
        assert L.lib().clothb200_launch_count() - n0 == 4      # schedule, sort, queue init, the persistent grid
    finally:
        L.check(L.lib().clothb200_debug_set_slicing(0, 0), "debug_set_slicing")
    f = bc.flags.cpu().numpy()
    assert (bc.sim_steps.cpu().numpy() == 0).all() and ((f & L.FLAG_NOGRAB) != 0).all()
    assert np.array_equal(bc.coverage.cpu().numpy(), mcov) and _bits_equal(bc.variance_inv.cpu().numpy(), mvinv)
    assert np.array_equal((f & L.FLAG_OOB) != 0, moob)


# ---------------------------------------------------------------------------------------------- 3. after real actions
def _aimed(bc, n, W, rng):
    pos = bc.pos[:, :, :3].double().cpu().numpy()
    a = rng.uniform(-1, 1, size=(n, 4))
    a[:, :2] = (pos[np.arange(n), rng.randint(0, W * W, size=n), :2] - 0.5) * 2
    return np.clip(a, -1, 1)


@pytest.mark.parametrize("W,mode", [(25, "ref"), (64, "col")])
def test_f32_actions_measure_as_the_oracle_on_their_state(W, mode):
    """After f32 actions the reported coverage and OOB flag are the oracle's on the f32 state the step returned, and
    variance_inv the restated kernel order on it - bit for bit."""
    L = _L()
    P, _ = _params(W)
    n, steps = (16, 2) if W == 25 else (8, 2)
    if W == 64:
        P.thickness = 0.006; P.reserved0 = 2             # bench.py config 4
    bc = _bc(P, n, "f32", L.MODE_COLOURED if mode == "col" else L.MODE_REFERENCE_ORDER)
    if W == 25:
        pool = load_golden("bench_pool_t1.npz")
        for e in range(n):
            bc.set_state(pool["pos"][e], pool["prev"][e], env=e)
    rng = np.random.RandomState(11 + W)
    gripped = 0
    for t in range(steps):
        out = {"sim_steps": np.zeros(n, np.int32), "coverage": np.zeros(n), "variance_inv": np.zeros(n),
               "flags": np.zeros(n, np.int32)}
        bc.step_host(_aimed(bc, n, W, rng), out)
        gripped += int((out["sim_steps"] > 0).sum())
        for e in range(n):
            s = _stored_back(bc, e)
            c, o = _oracle(W, s)
            assert out["coverage"][e] == c, (t, e, out["coverage"][e], c)
            assert _bits_equal(out["variance_inv"][e], variance_inv_kernel_order(s[:, 2], _nt(W))[0]), (t, e)
            assert bool(out["flags"][e] & L.FLAG_OOB) == o, (t, e)
    assert gripped >= n


# ---------------------------------------------------------------------------------------------- 4. bookkeeping
def _rect(W, X):
    """A grid on [0, X] x [0, 1]: hull area X exactly (shoelace 0.5 * (X*1 + X*1) from the corner (0, 0))."""
    g = _grid(W)
    g[:, 0] = g[:, 0] * X
    g[:, 2] = 0.05
    return g


def _run_book(dt, states, **kw):
    """step_plans with nothing-gripped plans and the bookkeeping pointers set."""
    L = _L()
    W = 25
    P, _ = _params(W)
    P.reward_type = kw.pop("reward_type", 0)
    initialize = kw.pop("initialize", False)
    bc = _bc(P, len(states), dt)
    _load(bc, states)
    bc.num_steps.fill_(kw.pop("num_steps", 0)); bc.num_sim_steps.fill_(7); bc.prev_coverage.fill_(kw.pop("prev_cov", 0.25))
    bc.reward.fill_(-9.0); bc.done.fill_(-1); bc.coverage.fill_(-7.0)
    assert not kw
    plans = _plans(len(states))
    host = torch.frombuffer(bytearray(bytes(plans)), dtype=torch.uint8).reshape(len(states), C.sizeof(L.Plan))
    bc.plans.copy_(host)
    io = bc.io(measure=True, bookkeeping=True, obs=False)
    L.check(bc._f("clothb200_step_plans")(C.byref(P), bc.mode, bc.n_env, C.c_void_p(bc.plans.data_ptr()), C.byref(io),
                                          int(initialize), bc.stream), "step_plans")
    torch.cuda.synchronize()
    out = {k: getattr(bc, k).cpu().numpy().copy() for k in ("coverage", "reward", "done", "num_steps", "num_sim_steps",
                                                              "prev_coverage", "sim_steps", "flags")}
    assert (out["sim_steps"] == 0).all() and ((out["flags"] & L.FLAG_NOGRAB) != 0).all()
    return P, out


def _reward(cov, prevc, reward_abs):
    """cloth_kernels.cuh's bookkeeping for an in-bounds, untorn cloth whose grip caught nothing, in its order."""
    rew = 0.0
    rew += -0.01
    if cov > 0.92:
        rew += 5.0
    rew += 0.0
    rew += cov if reward_abs else cov - prevc
    return rew


def _cov92(dt):
    """Widths X around 0.92 for the rectangle rows: (X, X > 0.92).  f64: 0.92 itself and both neighbours; f32: the
    f32 values on either side of the double 0.92 (none equals it)."""
    if dt == "f64":
        return [(np.nextafter(0.92, 0.0), False), (0.92, False), (np.nextafter(0.92, 1.0), True)]
    up = np.float32(0.92)
    if float(up) < 0.92:
        up = np.nextafter(up, np.float32(1))
    down = np.nextafter(up, np.float32(0))
    assert float(down) < 0.92 < float(up)
    return [(float(down), False), (float(up), True)]


@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_bonus_and_done_at_coverage_092(dt):
    cases = _cov92(dt)
    states = [("rect%r" % X, _stored(_rect(25, X), dt)) for X, _ in cases]
    P, out = _run_book(dt, states, num_steps=0, prev_cov=0.25)
    for e, (X, above) in enumerate(cases):
        cov = out["coverage"][e]
        assert cov == float(np.float64(X)) and cov == _oracle(25, states[e][1])[0], (X, cov)
        assert (cov > 0.92) == above
        assert out["reward"][e] == _reward(cov, 0.25, False), (X, out["reward"][e])
        assert out["done"][e] == int(above), (X, out["done"][e])
        assert out["prev_coverage"][e] == cov and out["num_steps"][e] == 1 and out["num_sim_steps"][e] == 7


@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_last_action_ends_the_episode(dt):
    L = _L()
    P, _ = _params(25)
    st = [("rect", _stored(_rect(25, 0.5), dt))]
    for preset, done in ((P.max_actions - 1, 1), (P.max_actions - 2, 0)):
        _, out = _run_book(dt, st, num_steps=preset)
        assert out["num_steps"][0] == preset + 1 and out["done"][0] == done, (preset, out["done"][0])
        assert out["reward"][0] == _reward(out["coverage"][0], 0.25, False)
    assert L.FLAG_NOGRAB


@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_reward_type_coverage_keeps_prev_coverage(dt):
    cases = _cov92(dt)
    states = [("rect%r" % X, _stored(_rect(25, X), dt)) for X, _ in cases]
    _, out = _run_book(dt, states, reward_type=1, prev_cov=0.375)
    for e, (X, above) in enumerate(cases):
        cov = out["coverage"][e]
        assert out["reward"][e] == _reward(cov, 0.375, True) and out["done"][e] == int(above), X
        assert out["prev_coverage"][e] == 0.375


@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_initialize_writes_coverage_but_no_bookkeeping(dt):
    states = [("rect", _stored(_rect(25, 0.75), dt))]
    _, out = _run_book(dt, states, initialize=True, num_steps=3, prev_cov=0.125)
    assert out["coverage"][0] == 0.75
    assert out["reward"][0] == -9.0 and out["done"][0] == -1 and out["num_steps"][0] == 3
    assert out["num_sim_steps"][0] == 7 and out["prev_coverage"][0] == 0.125


def test_nothing_gripped_costs_a_hundredth():
    for dt in ("f32", "f64"):
        states = [("rect", _stored(_rect(25, 0.5), dt))]
        _, out = _run_book(dt, states, prev_cov=0.5)
        assert out["reward"][0] == -0.01 + 0.0 + (0.5 - 0.5) and out["reward"][0] == -0.01


# ---------------------------------------------------------------------------------------------- 5. grip boundary
def _fma(a, b, c):
    """a*b + c rounded once (exact rational arithmetic; int / int true division rounds correctly)."""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def _verdicts(px, py, x, y, r):
    dx, dy = px - x, py - y
    return (dx * dx + dy * dy < r, _fma(dx, dx, dy * dy) < r, _fma(dy, dy, dx * dx) < r)


def _boundary_cases(r, count, seed):
    """(px, py, x, y): an f32 point and a double grip point whose plain test differs from a fused one."""
    rng = np.random.RandomState(seed)
    out = []
    while len(out) < count:
        px, py = (float(np.float32(v)) for v in rng.uniform(0.3, 0.7, 2))
        th = rng.uniform(0, 2 * np.pi)
        x0, y0 = px + math.sqrt(r) * math.cos(th), py + math.sqrt(r) * math.sin(th)
        for _ in range(40):
            x = x0 + rng.randint(-6, 7) * np.spacing(x0)
            y = y0 + rng.randint(-6, 7) * np.spacing(y0)
            v = _verdicts(px, py, x, y, r)
            if v[0] != v[1] or v[0] != v[2]:
                out.append((px, py, float(x), float(y)))
                break
    return out


def _lonely_point(W, px, py, far=(0.05, 0.05)):
    """A cloth at z = 0 packed into a small grid at `far`, except point 0 at (px, py)."""
    s = _grid(W) * 0.02
    s[:, 0] += far[0]; s[:, 1] += far[1]
    s[0, :2] = (px, py)
    return s


def _oracle_grip(W, s, x, y, r, force=False):
    o = OracleCloth(_oparams(W))
    o.set_state(s, s, np.zeros(len(s), np.uint8))
    o.grab_top(x, y, r)
    while force and len(o.grabbed) == 0:
        r += 0.02
        o.grab_top(x, y, r)
    return sorted(set(o.grabbed.tolist()))


@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_grab_top_on_the_radius_boundary(dt):
    """grab_top standalone and at the start of a step grips the oracle's set, where a fused multiply-add would not."""
    W = 25
    P, _ = _params(W)
    r = P.grip_radius
    cases = _boundary_cases(r, 256, 5)
    assert sum(_verdicts(*c, r)[0] for c in cases) not in (0, len(cases))   # both verdicts are exercised
    states = [("grip%d" % i, _stored(_lonely_point(W, px, py), dt)) for i, (px, py, _, _) in enumerate(cases)]
    exp = [_oracle_grip(W, s, x, y, r) for (_, s), (_, _, x, y) in zip(states, cases)]
    assert all(e in ([], [0]) for e in exp)
    n = len(states)
    # standalone: clothb200_grab_top with one grip point per cloth
    bc = _bc(P, n, dt)
    _load(bc, states)
    xy = torch.tensor([[c[2], c[3]] for c in cases], dtype=torch.float64, device="cuda")
    io = bc.io(measure=False, bookkeeping=False, obs=False)
    _L().check(bc._f("clothb200_grab_top")(C.byref(P), n, C.c_void_p(xy.data_ptr()), r, C.byref(io), bc.stream), "grab_top")
    torch.cuda.synchronize()
    got = [bc.grabbed_set(e).tolist() for e in range(n)]
    bad = [(i, cases[i], got[i], exp[i]) for i in range(n) if got[i] != exp[i]]
    assert not bad, ("grab_top", dt, len(bad), bad[:8])
    # at the start of a step
    bc = _bc(P, n, dt)
    _load(bc, states)
    plans = _plans(n)
    for p, (_, _, x, y) in zip(plans, cases):
        p.gx, p.gy = x, y
    bc.step_plans(plans)
    torch.cuda.synchronize()
    got = [bc.grabbed_set(e).tolist() for e in range(n)]
    ng = bc.n_grabbed.cpu().numpy()
    bad = [(i, cases[i], got[i], exp[i]) for i in range(n) if got[i] != exp[i] or ng[i] != len(exp[i])]
    assert not bad, ("step", dt, len(bad), bad[:8])


@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_force_grab_radius_grows_onto_the_boundary(dt):
    """force_grab widens the radius by 0.02 until something is gripped.  The designed point sits on the boundary of
    the third radius and a second point between the third and the fourth: the gripped set is {p} or {p, q} as the
    oracle's rounded test decides."""
    W = 25
    P, _ = _params(W)
    P.force_grab = 1
    r3 = P.grip_radius + 0.02 + 0.02
    r4 = r3 + 0.02
    cases = _boundary_cases(r3, 96, 9)
    states, exp = [], []
    for i, (px, py, x, y) in enumerate(cases):
        s = _lonely_point(W, px, py, far=(x + 0.9, y + 0.9))
        d = math.sqrt((r3 + r4) / 2)                   # q: gripped at r4, not at r3
        s[1, :2] = (x + d * math.cos(0.3), y + d * math.sin(0.3))
        s = _stored(s, dt)
        states.append(("force%d" % i, s))
        exp.append(_oracle_grip(W, _flush(s, dt), x, y, P.grip_radius, force=True))
    assert {tuple(e) for e in exp} == {(0,), (0, 1)}, {tuple(e) for e in exp}
    bc = _bc(P, len(states), dt)
    _load(bc, states)
    plans = _plans(len(states))
    for p, (_, _, x, y) in zip(plans, cases):
        p.gx, p.gy = x, y
    bc.step_plans(plans)
    torch.cuda.synchronize()
    got = [bc.grabbed_set(e).tolist() for e in range(len(states))]
    bad = [(i, cases[i], got[i], exp[i]) for i in range(len(states)) if got[i] != exp[i]]
    assert not bad, (dt, len(bad), bad[:8])
