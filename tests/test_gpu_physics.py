"""Per-environment material (ClothB200Physics rows, the `_phys` entry points, BatchedClothEnv.set_physics).

- Identity: rows equal to the batch's ClothB200Params give the plain entry points' bits, every output, all four
  families, f32 and f64, reference order and coloured, 25x25 with and without a rest table, 64x64 coloured, W = 16.
- f64 against the oracle, bit for bit: 16 crumpled tier-1 states with their own materials, 3 aimed actions, each
  environment against OracleCloth(params=<its material>), reference order and coloured.  Environment 15 tears while
  its neighbours do not; environment 0 (plane_friction < 1) differs from the same run at friction 1.
- f32 without a tolerance: environment e of a mixed batch equals a plain batch whose params carry e's material.
- Independence, time slicing (parked cloths take their row again on resume), invalid device rows, and whole
  BatchedClothEnv episodes (tier 1/2/3) against single-env ClothEnv instances whose cfg carries the material.
"""
import multiprocessing as mp
import os

import numpy as np
import pytest

from conftest import load_golden

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle.oracle import OracleCloth, params_from_cfg as oracle_params  # noqa: E402  (checker only)

F32, F64 = torch.float32, torch.float64
FIELDS = ("density", "ks", "damping", "plane_friction", "tear_thresh", "gravity")
# a material in the drawn ranges under which pool state 15 tears in the first action below (found on the CPU oracle)
TEARING = {"density": 400.0, "ks": 5000.0, "damping": 0.0, "plane_friction": 0.3, "tear_thresh": 1.3, "gravity": -12.0}


def _pool():
    g = load_golden("bench_pool_t1.npz")
    return {k: g[k] for k in g.files}


POOL = None


def pool():
    global POOL
    if POOL is None:
        POOL = _pool()
    return POOL


def _params(W=25):
    from gym_cloth_b200 import lib as L
    P = L.default_params()
    P.num_width_points = W; P.num_height_points = W
    if W != 25:
        P.thickness = 0.02 * 24 / (W - 1)
    return P


def _bc(P, n, dtype, mode=0, exact_rest=None):
    from gym_cloth_b200.batched import BatchedCloth
    return BatchedCloth(P, n, dtype=dtype, mode=mode, exact_rest=exact_rest)


def _draw(n, seed=7):
    """Materials of the ranges the feature is meant for: density and ks x[0.5, 2] of the defaults, damping [0, 5],
    plane_friction [0.3, 1], tear_thresh [1.3, 3], gravity [-12, -7]; row 15 = TEARING."""
    rng = np.random.RandomState(seed)
    m = {"density": 200.0 * rng.uniform(0.5, 2, n), "ks": 10000.0 * rng.uniform(0.5, 2, n), "damping": rng.uniform(0, 5, n),
         "plane_friction": rng.uniform(0.3, 1, n), "tear_thresh": rng.uniform(1.3, 3, n), "gravity": rng.uniform(-12, -7, n)}
    if n > 15:
        for k, v in TEARING.items():
            m[k][15] = v
    return m


def _row(m, e):
    return {k: float(m[k][e]) for k in FIELDS}


def _aimed(rng, pos):
    """bench.py's touch_cloth actions: raw U[-1,1]^4 with the grip aimed at a random mesh point of each cloth."""
    a = rng.uniform(-1, 1, size=(len(pos), 4))
    pick = rng.randint(0, pos.shape[1], size=len(pos))
    a[:, :2] = (pos[np.arange(len(pos)), pick, :2] - 0.5) * 2
    return a


def _load_pool(bc, n):
    p = pool()
    for e in range(n):
        bc.set_state(p["pos"][e], p["prev"][e], env=e)
    bc.prev_coverage.copy_(torch.from_numpy(p["start_coverage"][:n].copy()))


def _outs(bc):
    torch.cuda.synchronize()
    return {k: getattr(bc, k).clone().cpu().numpy() for k in ("pos", "prev", "flags", "sim_steps", "n_grabbed", "grab_mask",
                                                                  "coverage", "variance_inv", "obs", "reward", "done",
                                                                  "num_steps", "num_sim_steps")}


def _assert_equal(a, b, keys=None, what=""):
    for k in (keys or a):
        assert np.array_equal(a[k], b[k], equal_nan=True), (what, k)


def _set_rows(bc, m, envs=None):
    bc.set_physics(envs=envs, **m)


# ---------------------------------------------------------------------------------------------- 1. identity
IDENTITY = [  # (dtype, mode, W, exact_rest)
    (F64, 0, 25, True), (F64, 1, 25, True), (F64, 0, 16, True),
    (F32, 0, 25, False), (F32, 0, 25, True), (F32, 1, 25, False), (F32, 1, 64, False), (F32, 0, 16, False),
]


@pytest.mark.parametrize("dtype,mode,W,exact", IDENTITY)
def test_identity_rows_give_the_plain_bits(dtype, mode, W, exact):
    from gym_cloth_b200 import lib as L
    n = 16 if W != 64 else 4
    P = _params(W)
    a, b = _bc(P, n, dtype, mode, exact), _bc(P, n, dtype, mode, exact)
    b.set_physics(**L.physics_of(P))                     # every row = the batch's own material
    assert b.physics is not None
    rng = np.random.RandomState(5)
    if W == 25:
        _load_pool(a, n); _load_pool(b, n)
        pos = pool()["pos"][:n]
    else:
        # the flat grid, crumpled by a first action through the plain entry point on both
        pos = a.pos[:, :, :3].double().cpu().numpy()
        acts = _aimed(rng, pos)
        for c in (a, b):
            saved, c.physics = c.physics, None
            c.step_host(acts, {})
            c.physics = saved
        pos = a.pos[:, :, :3].double().cpu().numpy()
    # step_plans (host decode), step_actions (device decode), update_n, step_host
    acts = _aimed(rng, pos)
    for c in (a, b):
        c.step_plans(c.decode_host(acts))
    _assert_equal(_outs(a), _outs(b), what="step_plans")
    assert (_outs(a)["sim_steps"] > 0).any()
    acts = torch.from_numpy(_aimed(rng, a.pos[:, :, :3].double().cpu().numpy())).to("cuda", dtype)
    for c in (a, b):
        c.step_actions(acts)
    _assert_equal(_outs(a), _outs(b), what="step_actions")
    for c in (a, b):
        c.update(7, measure=True)
    _assert_equal(_outs(a), _outs(b), what="update_n")
    acts = _aimed(rng, a.pos[:, :, :3].double().cpu().numpy())
    ho = [{"obs": np.zeros((n, 3 * P.num_width_points ** 2), np.float32 if dtype == F32 else np.float64),
           "reward": np.zeros(n), "done": np.zeros(n, np.int32), "coverage": np.zeros(n), "variance_inv": np.zeros(n),
           "flags": np.zeros(n, np.int32), "sim_steps": np.zeros(n, np.int32)} for _ in range(2)]
    a.step_host(acts, ho[0]); b.step_host(acts, ho[1])
    _assert_equal(ho[0], ho[1], what="step_host host arrays")
    _assert_equal(_outs(a), _outs(b), what="step_host")


# ---------------------------------------------------------------------------------------------- 2. f64 vs oracle
def _oparams(m):
    OP = oracle_params(None)
    for k, v in m.items():
        setattr(OP, k, v)
    return OP


def _oracle_run(job):
    """Whole actions of the oracle from one pool state under one material (run in a forked worker)."""
    e, m, acts, mode = job
    p = pool()
    OP = _oparams(m)
    o = OracleCloth(OP, mode=mode)
    o.set_state(p["pos"][e], p["prev"][e], np.zeros(625, np.uint8))
    res = []
    for act in acts:
        k = OracleCloth(OP, mode=mode)                 # the grip list after the grab (a torn cloth keeps its old grip)
        k.set_state(*o.get_state(), grabbed=o.grabbed)
        plan = k.decode(act)
        k.grab_top(plan.gx, plan.gy)
        grab_list = sorted(set(k.grabbed.tolist()))
        try:
            nupd, ng, _ = o.step_action(act)
        except ZeroDivisionError:
            res.append({"bad": True})
            break
        pos, prev, pin = o.get_state()
        res.append({"bad": False, "nupd": nupd, "ng": ng, "grab_list": grab_list, "pos": pos, "prev": prev, "pin": pin,
                    "tear": o.tear, "oob": o.out_of_bounds(), "coverage": o.coverage()})
    return res


def _oracle_map(jobs):
    from oracle import oracle as O
    O.lib()                                   # built and loaded before the fork
    pool()
    with mp.get_context("fork").Pool(max(1, min(len(jobs), os.cpu_count() or 1))) as pl:
        return pl.map(_oracle_run, jobs, chunksize=1)


@pytest.mark.parametrize("mode", ["reference_order", "coloured"])
def test_f64_mixed_materials_match_the_oracle(mode):
    from gym_cloth_b200 import lib as L
    n = 16
    m = _draw(n)
    bc = _bc(_params(), n, F64, mode=L.MODE_COLOURED if mode == "coloured" else 0)
    _load_pool(bc, n)
    _set_rows(bc, m)
    rng = np.random.RandomState(3)
    acts, pos = [], pool()["pos"][:n]
    gpu = []
    for step in range(3):
        a = _aimed(rng, pos)
        acts.append(a)
        out = {"sim_steps": np.zeros(n, np.int32), "coverage": np.zeros(n), "flags": np.zeros(n, np.int32)}
        bc.step_host(a, out)
        torch.cuda.synchronize()
        gpu.append({"out": out, "states": [bc.get_state(e) for e in range(n)], "ngrab": bc.n_grabbed.cpu().numpy().copy(),
                    "mask": [bc.grabbed_set(e).tolist() for e in range(n)]})
        pos = np.stack([s[0] for s in gpu[-1]["states"]])
    jobs = [(e, _row(m, e), [acts[s][e] for s in range(3)], mode) for e in range(n)]
    fric1 = dict(_row(m, 0), plane_friction=1.0)
    jobs.append((0, fric1, [acts[s][0] for s in range(3)], mode))
    res = _oracle_map(jobs)
    for e in range(n):
        for s, r in enumerate(res[e]):
            g = gpu[s]
            if r["bad"]:
                assert g["out"]["flags"][e] & L.FLAG_BADSTATE, (e, s)
                break
            gp, gq, gpin, _ = g["states"][e]
            assert g["out"]["sim_steps"][e] == r["nupd"], (e, s)
            assert g["ngrab"][e] == r["ng"] and g["mask"][e] == r["grab_list"], (e, s)
            flags = (L.FLAG_TEAR if r["tear"] else 0) | (L.FLAG_OOB if r["oob"] else 0) | (L.FLAG_NOGRAB if r["ng"] == 0 else 0)
            assert g["out"]["flags"][e] == flags, (e, s, g["out"]["flags"][e], flags)
            assert np.array_equal(gp, r["pos"]) and np.array_equal(gq, r["prev"]), (e, s, np.abs(gp - r["pos"]).max())
            assert np.array_equal(gpin, r["pin"].astype(bool)), (e, s)
            assert abs(g["out"]["coverage"][e] - r["coverage"]) <= 1e-12, (e, s)
    # reference order: environment 15 tears in the first action while its neighbours do not (the coloured update
    # takes another path through the same material, and that cloth does not tear there)
    if mode == "reference_order":
        assert gpu[0]["out"]["flags"][15] & L.FLAG_TEAR
        assert not gpu[0]["out"]["flags"][14] & L.FLAG_TEAR
        assert sum(bool(f & L.FLAG_TEAR) for f in gpu[0]["out"]["flags"][:15]) < 15
    # environment 0 has plane_friction < 1 (fric1 != 0): friction 1 gives another result
    assert m["plane_friction"][0] < 1.0
    last = [r for r in res[n] if not r["bad"]][-1]
    assert not np.array_equal(gpu[len(res[n]) - 1]["states"][0][0], last["pos"])


# ---------------------------------------------------------------------------------------------- 3. f32 without a tolerance
@pytest.mark.parametrize("W,mode,exact", [(25, 0, False), (25, 0, True), (64, 1, False)])
def test_f32_mixed_batch_equals_plain_batches(W, mode, exact):
    n = 16
    m = _draw(n, seed=11)
    P = _params(W)
    mixed = _bc(P, n, F32, mode, exact)
    rng = np.random.RandomState(9)
    if W == 25:
        _load_pool(mixed, n)
        pos = pool()["pos"][:n]
    else:
        pos = mixed.pos[:, :, :3].double().cpu().numpy()
    acts = [_aimed(rng, pos)]
    _set_rows(mixed, m)
    mixed.step_host(acts[0], {})
    acts.append(_aimed(rng, mixed.pos[:, :, :3].double().cpu().numpy()))
    mixed.step_host(acts[1], {})
    got = _outs(mixed)
    assert (got["sim_steps"] > 0).any()
    for e in range(n):
        Pe = _params(W)
        for k in FIELDS:
            setattr(Pe, k, float(m[k][e]))
        plain = _bc(Pe, n, F32, mode, exact)
        if W == 25:
            _load_pool(plain, n)
        for a in acts:
            plain.step_host(a, {})
        ref = _outs(plain)
        for k in ref:
            assert np.array_equal(got[k][e], ref[k][e]), (e, k)


# ---------------------------------------------------------------------------------------------- 4. independence
def test_changing_one_material_changes_only_that_environment():
    n = 16
    m = _draw(n, seed=13)
    outs = []
    for damping3 in (m["damping"][3], m["damping"][3] + 1.5):
        bc = _bc(_params(), n, F32)
        _load_pool(bc, n)
        mm = {k: v.copy() for k, v in m.items()}
        mm["damping"][3] = damping3
        _set_rows(bc, mm)
        bc.step_host(_aimed(np.random.RandomState(2), pool()["pos"][:n]), {})
        outs.append(_outs(bc))
    a, b = outs
    assert not np.array_equal(a["pos"][3], b["pos"][3])
    for e in range(n):
        if e != 3:
            for k in a:
                assert np.array_equal(a[k][e], b[k][e]), (e, k)


# ---------------------------------------------------------------------------------------------- 5. time slicing
@pytest.mark.parametrize("dtype,mode", [(F64, 0), (F32, 0), (F32, 1)])
def test_time_sliced_mixed_batch_equals_unsliced(dtype, mode):
    from gym_cloth_b200 import lib as L
    from test_gpu_slicing import queue_parks
    n = 16
    m = _draw(n, seed=17)
    lib = L.lib()
    runs, parks = [], []
    for sliced in (False, True):
        bc = _bc(_params(), n, dtype, mode)
        _load_pool(bc, n)
        _set_rows(bc, m)
        bc.time_slice = sliced
        rng = np.random.RandomState(4)
        if sliced:
            lib.clothb200_debug_set_slicing(3, 37)     # three resident cloths, slices of 37 substeps
        try:
            outs = []
            for _ in range(2):
                a = torch.from_numpy(_aimed(rng, bc.pos[:, :, :3].double().cpu().numpy())).to("cuda", dtype)
                bc.step_actions(a)
                outs.append(_outs(bc))
                if sliced:
                    parks.append(queue_parks(bc))
        finally:
            lib.clothb200_debug_set_slicing(0, 0)
        runs.append(outs)
    for s in range(2):
        _assert_equal(runs[0][s], runs[1][s], what="sliced step %d" % s)
    assert sum(parks) > 0, parks


# ---------------------------------------------------------------------------------------------- 6. invalid device rows
@pytest.mark.parametrize("dtype", [F32, F64])
def test_invalid_rows_are_bad_actions(dtype):
    import ctypes as C
    from gym_cloth_b200 import lib as L
    n = 8
    m = _draw(n, seed=19)
    bad = {2: ("density", 0.0), 5: ("ks", float("nan"))}
    acts = _aimed(np.random.RandomState(6), pool()["pos"][:n])
    res = []
    for with_bad in (False, True):
        bc = _bc(_params(), n, dtype)
        _load_pool(bc, n)
        _set_rows(bc, m)
        if with_bad:
            for e, (k, v) in bad.items():
                bc.physics[e, FIELDS.index(k)] = v
        bc.flags.zero_()
        plans = bc.decode_host(acts)
        bc.plans.copy_(torch.frombuffer(bytearray(bytes(plans)), dtype=torch.uint8).reshape(n, -1))
        io = bc.io()
        rc = getattr(bc.L, "clothb200_step_plans_phys" + bc.sfx)(C.byref(bc.P), 0, n, C.c_void_p(bc.plans.data_ptr()), C.byref(io),
                                                                0, C.c_void_p(bc.physics.data_ptr()), bc.stream)
        assert rc == 0
        torch.cuda.synchronize()                                  # no CUDA error behind
        step = _outs(bc)
        bc.update(5)
        torch.cuda.synchronize()
        res.append((step, _outs(bc)))
    (ok_step, ok_upd), (bad_step, bad_upd) = res
    p = pool()
    for e in range(n):
        if e in bad:
            assert (bad_step["flags"][e] & ~L.FLAG_OOB) == (L.FLAG_BADSTATE | L.FLAG_NOGRAB), e
            assert bad_step["sim_steps"][e] == 0 and bad_step["n_grabbed"][e] == 0
            assert bad_step["reward"][e] == -0.01 + (bad_step["coverage"][e] - p["start_coverage"][e])
            assert np.array_equal(bad_step["pos"][e][:, :3], p["pos"][e].astype(bad_step["pos"].dtype))
            assert np.array_equal(bad_step["prev"][e][:, :3], p["prev"][e].astype(bad_step["prev"].dtype))
            assert bad_upd["flags"][e] & L.FLAG_BADSTATE and bad_upd["sim_steps"][e] == 0
            assert np.array_equal(bad_upd["pos"][e], bad_step["pos"][e])
        else:
            for k in ok_step:
                assert np.array_equal(ok_step[k][e], bad_step[k][e]), (e, k)
                assert np.array_equal(ok_upd[k][e], bad_upd[k][e]), (e, k)


# ---------------------------------------------------------------------------------------------- 7. environment level
@pytest.mark.parametrize("tier", [1, 2, 3])
def test_env_episodes_match_single_envs_with_that_cfg(tier):
    from gym_cloth_b200 import cfg_path
    from gym_cloth_b200.envs import BatchedClothEnv, ClothEnv
    from gym_cloth_b200.envs.cloth_env import load_cfg
    n, seed = 3, 31
    m = _draw(n, seed=23 + tier)
    m["tear_thresh"] = np.maximum(m["tear_thresh"], 2.0)
    # dom_rand_draws: the batch replays the per-reset draws the single-env facade replays, so the generators compare
    benv = BatchedClothEnv(cfg_path(tier), n, dtype="f64", seed=seed, physics=m, dom_rand_draws=True)
    ph = benv.get_physics()
    for k in FIELDS:
        assert np.array_equal(ph[k], m[k]), k
    bobs = [benv.reset().clone().cpu().numpy()]
    brng = np.random.RandomState(41)
    acts = [brng.uniform(-1, 1, size=(n, 4)) * np.array([0.6, 0.6, 1, 1]) for _ in range(2)]
    bres = []
    for a in acts:
        obs, rew, done, info = benv.step(a)
        bres.append((np.array(obs), np.array(rew), np.array(done), {k: (v.cpu().numpy() if torch.is_tensor(v) else np.array(v))
                                                                     for k, v in info.items()}))
    bstate = [benv.cloth.get_state(e) for e in range(n)]
    assert np.array_equal(benv.get_physics()["ks"], m["ks"])         # kept across reset()
    for e in range(n):
        cfg = load_cfg(cfg_path(tier))
        for k in ("density", "ks", "damping", "plane_friction", "tear_thresh"):
            cfg["cloth"][k] = float(m[k][e])
        env = ClothEnv(cfg, dtype="f64")
        env._b.P.gravity = float(m["gravity"][e])                    # Cloth's gravity argument (cloth.pyx:24-26)
        env.seed(seed + e)
        obs0 = env.reset()
        assert np.array_equal(obs0, bobs[0][e]), e
        for s, a in enumerate(acts):
            obs, rew, done, info = env.step(a[e])
            bo, br, bd, bi = bres[s]
            assert np.array_equal(obs, bo[e]) and rew == br[e] and bool(done) == bool(bd[e]), (e, s)
            assert info["actual_coverage"] == bi["actual_coverage"][e] and info["variance_inv"] == bi["variance_inv"][e]
            assert info["have_tear"] == bool(bi["have_tear"][e]) and info["out_of_bounds"] == bool(bi["out_of_bounds"][e])
        sp, sq, spin, sg = env._b.cloth.get_state(0)
        bp, bq, bpin, bg = bstate[e]
        assert np.array_equal(sp, bp) and np.array_equal(sq, bq) and np.array_equal(spin, bpin) and np.array_equal(sg, bg)
        a_st, b_st = env.np_random.get_state(), benv.rngs[e].get_state()
        assert np.array_equal(a_st[1], b_st[1]) and a_st[2:] == b_st[2:], e
