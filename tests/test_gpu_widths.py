"""The reference-order kernel away from its 25x25 / 128-thread configuration, against the oracle.

ClothCTA::ORDERED (the ordered scatter) holds only for the compile-time 25x25 grid run by four warps.  Every other grid
width (the runtime-width kernel), and any grid under CLOTHB200_NT=256, takes the unordered scatter and ranks the
members of each bucket back into point-index order (collide_buckets, order_bucket for piles of more than 32 points).
The limit pass has two exact strategies (queue replay and wavefront sweep) picked per substep.  The f64 build must
equal the oracle bit for bit on every one of these paths:

1. whole actions at W = 3 ... 55 (the smallest grid, the power-of-two cells 4, 7, 13, 49, both neighbours of 25 and
   the largest f64 grid one CTA's shared memory holds), thickness scaled to 0.02*24/(W-1);
2. piles of 33 to 300 points in one hash cell (each register / shared-memory replay at its boundary), at W = 25 and 40;
3. the CLOTHB200_NT and CLOTHB200_SWEEP_THRESH knobs, each in a child process (they are read once per process), and
   the README's claim that results never depend on them, bit for bit in f32 too;
4. f32 grids above the f64 limit, the shared-memory size clothb200_occupancy reports, and the refusal of grids that
   do not fit.

The device's profile counters (clothb200_debug_set_profile, [n_env][16]) show which paths ran: [5] piles of more than
32 points, [12] limit-queue pops, [13] springs the limit pass moved.  Oracle actions run in a fork pool over the host
cores, as scripts/fuzz_f64.py does.
"""
import ctypes as C
import functools
import json
import multiprocessing as mp
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import load_golden

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle.oracle import OracleCloth, params_from_cfg as oracle_params  # noqa: E402  (checker only)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64, F32 = torch.float64, torch.float32
WIDTHS = [3, 4, 7, 13, 16, 24, 26, 33, 40, 49, 55]
N_ENV, N_ACT = 8, 3
PROF_PILES, PROF_POPS, PROF_MOVES = 5, 12, 13


def _thickness(W):
    """Tier 1's ratio of collision threshold to grid spacing at every width."""
    return 0.02 * 24 / (W - 1)


def _oparams(W, ks=None, gravity=None):
    OP = oracle_params(None)
    OP.num_width_points = W; OP.num_height_points = W
    OP.thickness = _thickness(W)
    if ks is not None:
        OP.ks = ks
    if gravity is not None:
        OP.gravity = gravity
    return OP


def _params(W, ks=None, gravity=None):
    from gym_cloth_b200 import lib as L
    P = L.default_params()
    P.num_width_points = W; P.num_height_points = W
    P.thickness = _thickness(W)
    if ks is not None:
        P.ks = ks
    if gravity is not None:
        P.gravity = gravity
    return P, _oparams(W, ks, gravity)


def _bc(P, n, dtype=F64):
    from gym_cloth_b200 import lib as L
    from gym_cloth_b200.batched import BatchedCloth
    return BatchedCloth(P, n, dtype=dtype, mode=L.MODE_REFERENCE_ORDER)


class _Profile(object):
    """The device's per-environment counters of the launches run inside the block (each launch of fewer cloths than
    resident slots overwrites its environments' rows)."""

    def __init__(self, n):
        self.t = torch.zeros(n, 16, dtype=torch.int64, device="cuda")

    def __enter__(self):
        from gym_cloth_b200 import lib as L
        L.lib().clothb200_debug_set_profile(C.c_void_p(self.t.data_ptr()))
        return self

    def __exit__(self, *exc):
        from gym_cloth_b200 import lib as L
        torch.cuda.synchronize()
        L.lib().clothb200_debug_set_profile(None)

    def get(self):
        return self.t.cpu().numpy()


def _assert_same(bc, e, pos, prev, pin, what):
    gp, gq, gpin, _ = bc.get_state(e)
    assert np.array_equal(gp, pos), (what, e, np.abs(gp - pos).max())
    assert np.array_equal(gq, prev), (what, e, np.abs(gq - prev).max())
    assert np.array_equal(gpin, pin.astype(bool)), (what, e)


# ---------------------------------------------------------------------------------------------- oracle pool
def _oracle_action(job):
    """One whole action of the oracle from a given state (run in a forked worker)."""
    W, (pos, prev, pin, grabbed, tear), act = job
    OP = _oparams(W)
    # the grip list after the grab: a torn cloth is never released, so its old grip stays in it (as in the kernel)
    k = OracleCloth(OP)
    k.set_state(pos, prev, pin, grabbed=grabbed)
    plan = k.decode(act)
    k.grab_top(plan.gx, plan.gy)
    grab_list = k.grabbed.tolist()
    o = OracleCloth(OP)
    o.set_state(pos, prev, pin, grabbed=grabbed, tear=tear)
    try:
        nupd, ng, _ = o.step_action(act)
    except ZeroDivisionError:
        return {"bad": True}
    p, q, pn = o.get_state()
    return {"bad": False, "nupd": nupd, "ng": ng, "grab_list": grab_list, "pos": p, "prev": q, "pin": pn,
            "grabbed": o.grabbed, "tear": o.tear, "oob": o.out_of_bounds(), "coverage": o.coverage(),
            "variance_inv": o.variance_inv(), "counters": o.counters()}


def _oracle_map(jobs):
    from oracle import oracle as O
    O.lib()                                   # built and loaded before the fork
    with mp.get_context("fork").Pool(max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
        return pool.map(_oracle_action, jobs, chunksize=1)


def _empty_spot(pos, clearance):
    """An (x, y) in the unit square at least `clearance` from every point of the cloth in the plane, or None."""
    from scipy.spatial import cKDTree
    g = np.linspace(0.0, 1.0, 201)
    X, Y = np.meshgrid(g, g, indexing="ij")
    cand = np.stack([X.ravel(), Y.ravel()], -1)
    d, _ = cKDTree(pos[:, :2]).query(cand)
    i = int(np.argmax(d))
    return cand[i] if d[i] >= clearance else None


def _actions(W, t, states, nograb_done):
    """bench.py's touch_cloth draws, one seed per (width, environment, action), aimed at a random mesh point of each
    cloth.  Environment N_ENV-1 aims once at a spot no point is within grip range of: an action that grabs nothing."""
    acts = np.zeros((len(states), 4))
    for e, st in enumerate(states):
        rng = np.random.RandomState(100000 * W + 100 * e + t)
        a = rng.uniform(-1, 1, size=4)
        a[:2] = (st[0][rng.randint(0, len(st[0])), :2] - 0.5) * 2
        acts[e] = np.clip(a, -1, 1)
    if not nograb_done:
        spot = _empty_spot(states[-1][0], 0.06)        # the grip takes points with dx^2 + dy^2 < grip_radius = 0.003
        if spot is not None:
            acts[-1, :2] = spot * 2 - 1
            return acts, True
    return acts, False


def _check_action(bc, out, res, t):
    from gym_cloth_b200 import lib as L
    for e, r in enumerate(res):
        what = ("action", t, "env", e)
        if r["bad"]:
            assert out["flags"][e] & L.FLAG_BADSTATE, what
            continue
        assert out["sim_steps"][e] == r["nupd"], (what, out["sim_steps"][e], r["nupd"])
        assert bc.n_grabbed[e].item() == r["ng"] == len(r["grab_list"]), what
        assert bc.grabbed_set(e).tolist() == sorted(set(r["grab_list"])), what
        flags = (L.FLAG_TEAR if r["tear"] else 0) | (L.FLAG_OOB if r["oob"] else 0) | (L.FLAG_NOGRAB if r["ng"] == 0 else 0)
        assert out["flags"][e] == flags, (what, out["flags"][e], flags)
        _assert_same(bc, e, r["pos"], r["prev"], r["pin"], what)
        assert abs(out["coverage"][e] - r["coverage"]) <= 1e-12, what
        assert abs(out["variance_inv"][e] - r["variance_inv"]) <= 1e-12 * abs(r["variance_inv"]), what


@functools.lru_cache(maxsize=None)
def _widths_case(W):
    """N_ENV flat W x W cloths, N_ACT sequential aimed actions through step_host, every action compared with the
    oracle.  Returns the totals the assertions and the -s report use."""
    P, _ = _params(W)
    bc = _bc(P, N_ENV)
    pos0, prev0, pin0, _ = bc.get_state(0)
    states = [(pos0, prev0, pin0.astype(np.uint8), np.zeros(0, np.int32), False) for _ in range(N_ENV)]
    tot = {"W": W, "substeps": 0, "collide_hits": 0, "stretched": 0, "pops": 0, "moves": 0, "piles": 0, "nograb": 0}
    nograb_done = False
    for t in range(N_ACT):
        acts, aimed_off = _actions(W, t, states, nograb_done)
        nograb_done |= aimed_off
        out = {"sim_steps": np.zeros(N_ENV, np.int32), "coverage": np.zeros(N_ENV), "variance_inv": np.zeros(N_ENV),
               "flags": np.zeros(N_ENV, np.int32)}
        with _Profile(N_ENV) as prof:
            bc.step_host(acts, out)
        res = _oracle_map([(W, st, acts[e]) for e, st in enumerate(states)])
        _check_action(bc, out, res, t)
        pr = prof.get()
        tot["pops"] += int(pr[:, PROF_POPS].sum()); tot["moves"] += int(pr[:, PROF_MOVES].sum())
        tot["piles"] += int(pr[:, PROF_PILES].sum())
        for e, r in enumerate(res):
            if r["bad"]:
                continue
            tot["substeps"] += r["nupd"]
            tot["collide_hits"] += r["counters"]["collide_hits"]; tot["stretched"] += r["counters"]["stretched"]
            tot["nograb"] += r["ng"] == 0
            states[e] = (r["pos"], r["prev"], r["pin"], r["grabbed"], r["tear"])
    print("W=%d: %d substeps, oracle collide_hits %d stretched %d, device pops %d moves %d piles %d, %d grabbed nothing"
          % (W, tot["substeps"], tot["collide_hits"], tot["stretched"], tot["pops"], tot["moves"], tot["piles"], tot["nograb"]))
    return tot


# ---------------------------------------------------------------------------------------------- 1. widths
@pytest.mark.parametrize("W", WIDTHS)
def test_f64_widths_whole_actions_bit_exact(W):
    tot = _widths_case(W)
    assert tot["collide_hits"] > 0 and tot["stretched"] > 0, tot       # both Gauss-Seidel passes had work
    assert tot["moves"] > 0, tot
    assert tot["nograb"] >= 1, tot


def test_f64_widths_ran_a_pile():
    """At least one grid of 33 or more points a side piled more than 32 points into one cell during the actions."""
    piles = {W: _widths_case(W)["piles"] for W in WIDTHS if W >= 33}
    assert sum(piles.values()) > 0, piles


# ---------------------------------------------------------------------------------------------- 2. piles
PILES = (33, 64, 65, 128, 129, 200, 300)


def _pile_states(W):
    """Flat W x W cloths with points piled into hash cells at z in the second cell layer, where no cloth point lies.
    Spring stiffness and gravity are 0, so Verlet leaves the points where they are and the first substep hashes
    exactly these piles (with the default ks the springs fling a pile's points out of its cell before the hash).
    Returns (name, pos, pinned, {cell key: size}) per state."""
    cw = 3.0 / (W - 1)
    r, c = np.meshgrid(np.arange(W), np.arange(W), indexing="ij")
    flat = np.stack([r / (W - 1.0), c / (W - 1.0), np.zeros_like(r, float)], -1).reshape(-1, 3)
    rng = np.random.RandomState(W)
    i0 = W // 6

    def pile(p, idx, ci):
        centre = np.array([(ci + 0.5) * cw, (i0 + 0.5) * cw, 1.5 * cw])
        p[idx] = centre + rng.uniform(-1, 1, size=(len(idx), 3)) * (0.3 * cw)
        return 961 * ci + 31 * i0 + 1

    out = []
    for n in PILES:
        p = flat.copy()
        key = pile(p, rng.choice(W * W, n, replace=False), i0)
        out.append(("pile%d" % n, p, np.zeros(W * W, np.uint8), {key: n}))
    p = flat.copy()
    idx = rng.choice(W * W, 40 + 100, replace=False)
    ka = pile(p, idx[:40], i0); kb = pile(p, idx[40:], i0 + 1)
    out.append(("neighbours", p, np.zeros(W * W, np.uint8), {ka: 40, kb: 100}))
    p = flat.copy()
    idx = rng.choice(W * W, 90, replace=False)
    key = pile(p, idx, i0)
    pin = np.zeros(W * W, np.uint8); pin[idx[::4]] = 1
    out.append(("pinned", p, pin, {key: 90}))
    return out


def _cell_sizes(pos, W):
    cw = 3 * (1.0 / (W - 1))
    f = np.floor(pos / cw).astype(np.int64)
    keys, counts = np.unique(961 * f[:, 0] + 31 * f[:, 1] + f[:, 2], return_counts=True)
    return dict(zip(keys.tolist(), counts.tolist()))


@functools.lru_cache(maxsize=None)
def _piles_case(W):
    P, OP = _params(W, ks=0.0, gravity=0.0)
    states = _pile_states(W)
    bc = _bc(P, len(states))
    for e, (name, p, pin, sizes) in enumerate(states):
        have = _cell_sizes(p, W)
        assert all(have[k] == v for k, v in sizes.items()), (name, sizes)   # the piles are exactly as built
        bc.set_state(p, p, pin, env=e)
    with _Profile(len(states)) as prof:
        bc.update(3)
    pr = prof.get()
    hits = []
    for e, (name, p, pin, sizes) in enumerate(states):
        o = OracleCloth(OP)
        o.set_state(p, p, pin)
        o.update(3)
        c = o.counters()
        assert c["collide_hits"] > 0 and c["stretched"] > 0, (name, c)
        assert pr[e, PROF_PILES] >= len(sizes), (name, pr[e])
        op, oq, opin = o.get_state()
        _assert_same(bc, e, op, oq, opin, (W, name))
        hits.append(c["collide_hits"])
    print("W=%d piles: oracle collide_hits %s, device piles %s" % (W, hits, pr[:, PROF_PILES].tolist()))
    return {"piles": pr[:, PROF_PILES].tolist()}


@pytest.mark.parametrize("W", [25, 40])
def test_f64_piles_bit_exact(W):
    _piles_case(W)


# ---------------------------------------------------------------------------------------------- 3. knobs
def _f32_outputs():
    """f32 results for the knob comparison: 16 crumpled pool states at 25x25 with one aimed action each, and 4 cloths
    at 64x64 driven through two aimed actions from the flat grid (the first crumples them)."""
    from gym_cloth_b200 import lib as L
    out = {}
    pool = load_golden("bench_pool_t1.npz")
    runs = [(25, 16, 1), (64, 4, 2)]
    for W, n, steps in runs:
        P = L.default_params()
        P.num_width_points = W; P.num_height_points = W; P.thickness = _thickness(W)
        bc = _bc(P, n, F32)
        if W == 25:
            for e in range(n):
                bc.set_state(pool["pos"][e], pool["prev"][e], env=e)
        rng = np.random.RandomState(7 + W)
        for t in range(steps):
            pos = bc.pos[:, :, :3].double().cpu().numpy()
            a = rng.uniform(-1, 1, size=(n, 4))
            a[:, :2] = (pos[np.arange(n), rng.randint(0, W * W, size=n), :2] - 0.5) * 2
            host = {"sim_steps": np.zeros(n, np.int32), "coverage": np.zeros(n), "variance_inv": np.zeros(n),
                    "flags": np.zeros(n, np.int32)}
            bc.step_host(np.clip(a, -1, 1), host)
            for k, v in host.items():
                out["%d_%d_%s" % (W, t, k)] = v.copy()
            for k in ("pos", "prev", "n_grabbed", "grab_mask"):
                out["%d_%d_%s" % (W, t, k)] = getattr(bc, k).cpu().numpy()
    return out


# Each knob setting runs in a child process.  It checks the f64 cases against the oracle itself (an assertion fails
# the child), writes its f32 results and prints the summed device counters as the last line.
CHILD = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import test_gpu_widths as T
res = {"widths": {}, "piles": {}}
for W in (25, 40):
    res["widths"][W] = T._widths_case(W)
    if "piles" in sys.argv[3]:
        res["piles"][W] = T._piles_case(W)
if "f32" in sys.argv[3]:
    np.savez(sys.argv[2], **T._f32_outputs())
print(json.dumps(res))
"""

KNOBS = {
    "nt256": ({"CLOTHB200_NT": "256"}, "piles,f32"),
    "sweep1": ({"CLOTHB200_SWEEP_THRESH": "1"}, "f32"),
    "sweep0": ({"CLOTHB200_SWEEP_THRESH": "0"}, "f32"),
    "sweep1000000": ({"CLOTHB200_SWEEP_THRESH": "1000000"}, ""),
}
_CHILDREN = {}


def _child(name, tmp_path_factory):
    if name not in _CHILDREN:
        env_add, what = KNOBS[name]
        out = tmp_path_factory.mktemp(name) / "f32.npz"
        env = dict(os.environ, **env_add)
        for k in ("CLOTHB200_NT", "CLOTHB200_SWEEP_THRESH"):
            if k not in env_add:
                env.pop(k, None)
        r = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(out), what], env=env, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=1200)
        assert r.returncode == 0, (name, r.stdout[-6000:])
        print("child %s:\n%s" % (name, "\n".join(r.stdout.splitlines()[:-1])))
        res = json.loads(r.stdout.strip().splitlines()[-1])
        _CHILDREN[name] = (res, dict(np.load(out)) if "f32" in what else None)
    return _CHILDREN[name]


def test_knob_nt256_f64_unordered_path_bit_exact(tmp_path_factory):
    """W = 25 under 8 warps drops from the ordered to the unordered scatter inside the compile-time kernel."""
    res, _ = _child("nt256", tmp_path_factory)
    assert set(res["widths"]) == {"25", "40"} and set(res["piles"]) == {"25", "40"}


@pytest.mark.parametrize("thresh", [1, 0, 1000000])
def test_knob_sweep_threshold_f64_bit_exact(thresh, tmp_path_factory):
    res, _ = _child("sweep%d" % thresh, tmp_path_factory)
    for W, tot in res["widths"].items():
        if thresh == 1:
            assert tot["pops"] == 0 and tot["moves"] > 0, (W, tot)       # the sweep did all the work
        else:
            assert tot["pops"] > 0, (W, tot)                              # the queue replay ran


@functools.lru_cache(maxsize=None)
def _f32_default():
    return _f32_outputs()


@pytest.mark.parametrize("name,widths", [("nt256", (25, 64)), ("sweep1", (25,)), ("sweep0", (25,))])
def test_knobs_keep_f32_bits(name, widths, tmp_path_factory):
    """CLOTHB200_NT 128 vs 256 at 25x25 and 256 vs 512 at 64x64 (the defaults are 128 and 512), and the sweep threshold
    1 vs 0 vs the default at 25x25: the f32 build gives the same bits - state, substeps, grips, flags and coverage.
    The one exception is variance_inv under CLOTHB200_NT: it is a block-wide double sum whose order follows the thread
    count, so it may differ in the last bits (held to 1e-12 relative, the bound the f64 build keeps against np.var)."""
    _, got = _child(name, tmp_path_factory)
    ref = _f32_default()
    keys = [k for k in ref if int(k.split("_")[0]) in widths]
    assert keys
    differ = [k for k in keys if not np.array_equal(ref[k], got[k])]
    rel = max(float(np.max(np.abs(got[k] - ref[k]) / np.abs(ref[k]))) for k in keys if k.endswith("variance_inv"))
    print("%s: max relative variance_inv difference %.2e; arrays that differ: %s" % (name, rel, differ))
    if name.startswith("nt"):
        differ = [k for k in differ if not k.endswith("variance_inv")]
        assert rel <= 1e-12, (name, rel)
    assert not differ, (name, differ)


# ---------------------------------------------------------------------------------------------- 4. size limits
def _drive(bc, o):
    bc.grab_top((0.5, 0.5)); o.grab_top(0.5, 0.5)
    assert bc.n_grabbed[0].item() == len(o.grabbed) > 0
    for i in range(12):
        bc.adjust(0.0, 0.0, 0.0025); o.adjust(0.0, 0.0, 0.0025)
        bc.update(1); o.update(1)
    for i in range(6):
        bc.adjust(0.002, -0.001, 0.0); o.adjust(0.002, -0.001, 0.0)
        bc.update(1); o.update(1)


@pytest.mark.parametrize("W", [56, 65])
def test_f32_above_the_f64_limit_vs_oracle(W):
    """W = 65 has more than 4096 points: no sweep table, the queue replay does every limit pass."""
    P, OP = _params(W)
    bc = _bc(P, 2, F32)
    o = OracleCloth(OP)
    with _Profile(2) as prof:
        _drive(bc, o)
    pos, prev, pin, _ = bc.get_state(1)
    op, oq, opin = o.get_state()
    d = np.abs(pos - op).max()
    pr = prof.get()
    print("f32 %dx%d reference order, 18 substeps: max |dpos| %.3e, pops %d, moves %d, oracle %s"
          % (W, W, d, pr[1, PROF_POPS], pr[1, PROF_MOVES], o.counters()))
    assert d <= 5e-6 and np.array_equal(pin, opin.astype(bool))
    assert o.counters()["stretched"] > 0


def _smem_bytes(W, elem):
    """ClothCTA::smem_bytes with make_dev_params' hash sizing (cloth_kernels.cuh, cloth_device.cuh) for the
    reference-order kernel: away from the ordered 25x25 grid it has a counter block of 2*NCLS ints of its own."""
    N = W * W
    cells = (W + 2) // 3 + 1
    ts = 64
    while ts < 3 * cells * cells:
        ts <<= 1
    np2 = 1
    while np2 < N:
        np2 <<= 1
    while 4 * ts < np2:
        ts <<= 1
    ev_words = (6 * N + 31) // 32
    ps = 2 * ((N + 7) & ~7)
    ev = 4 * ((ev_words + 3) & ~3)
    cls = 0 if W == 25 else 8 * 34
    return 4 * elem * N * 2 + 8 * ts + 64 + 128 + 64 + max(ps, ev) + 2 * ps + cls + 16


SIZES = [("f64", 25, 48160, True), ("f64", 55, 228720, True), ("f64", 56, 236448, False), ("f32", 70, 203152, True),
         ("f32", 77, 258656, False)]


@pytest.mark.parametrize("dt,W,smem,fits", SIZES)
def test_occupancy_reports_the_shared_memory_of_one_cloth(dt, W, smem, fits):
    from gym_cloth_b200 import lib as L
    P, _ = _params(W)
    ctas, got, thr = C.c_int(0), C.c_int(0), C.c_int(0)
    L.check(L.lib().clothb200_occupancy(C.byref(P), int(dt == "f64"), C.byref(ctas), C.byref(got), C.byref(thr)), "occupancy")
    assert got.value == _smem_bytes(W, 8 if dt == "f64" else 4) == smem
    limit = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    print("%s %dx%d: %d B of shared memory, %d B per block on this device" % (dt, W, W, got.value, limit))
    assert (got.value <= limit) == fits


@pytest.mark.parametrize("dt,W", [("f64", 56), ("f32", 77)])
def test_grid_too_large_for_one_cta_is_refused(dt, W):
    """The step and the bare update return CLOTHB200_ERR_UNSUPPORTED and leave the state alone; the failed attribute
    call leaves no error behind for the next CUDA call of the process."""
    from gym_cloth_b200 import lib as L
    P, _ = _params(W)
    n = 2
    bc = _bc(P, n, F64 if dt == "f64" else F32)
    pos0, prev0 = bc.pos.clone(), bc.prev.clone()
    with pytest.raises(L.ClothB200Error) as ei:
        bc.step_host(np.array([[0.0, 0.0, 0.3, 0.2], [0.4, -0.2, -0.3, 0.1]]), {"sim_steps": np.zeros(n, np.int32)})
    assert ei.value.code == -4, str(ei.value)
    with pytest.raises(L.ClothB200Error) as ei:
        bc.update(1)
    assert ei.value.code == -4, str(ei.value)
    torch.cuda.synchronize()
    assert torch.equal(bc.pos, pos0) and torch.equal(bc.prev, prev0)
    # the process goes on: a PyTorch kernel and a cloth that fits
    x = torch.arange(1000, device="cuda", dtype=torch.float64).cumsum(0)
    torch.cuda.synchronize()
    assert x[-1].item() == 999 * 1000 / 2
    small, _ = _params(25)
    ok = _bc(small, 1, F64 if dt == "f64" else F32)
    ok.update(2)
    torch.cuda.synchronize()
