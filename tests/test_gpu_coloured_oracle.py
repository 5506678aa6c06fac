"""The graph-coloured kernels (CLOTHB200_MODE_COLOURED) against the oracle's coloured update (oracle_update_coloured).

f64 build, bit for bit (np.array_equal on positions, previous positions and pins).  The f64 kernels are built with
-fmad=false, the Jacobi collision sums each bucket in member-index order, and the springs of one colour class share no
point, so the parallel update is one sequential order of the same IEEE operations.

f32 build, within twice what was measured on an NVIDIA B200 (power limit 1000 W), the convention of
test_gpu_f32_contract.py.  Inputs are seeded and the kernels deterministic, so each value is one measurement:

  25x25, max |dpos| vs the coloured oracle           measured                        asserted
    phases.npz pull, substep 1 / 10 / 50              1.2e-7 / 6.4e-7 / 5.2e-6        2.4e-7 / 1.3e-6 / 1.1e-5
    App. D lift, substep 1 / 10 / 50                  2.0e-8 / 1.8e-7 / 1.7e-6        4e-8 / 3.6e-7 / 3.4e-6
    64 pool states x one action: identical substep counts and grabbed sets,
      |mean coverage difference|                      1.3e-3                          2.7e-3
      (max |dpos| 0.30 and max |coverage difference| 3.8e-2 over the 64: a whole action is chaotic, not asserted)
  64x64, thickness 0.006 (BASELINE config 4), relax_iters 1 and 2
    _drive schedule (18 substeps), max |dpos|         2.9e-7 / 3.7e-7                 7.4e-7
    one action on 3 cloths: identical substep counts, grab counts and grabbed sets,
      max |coverage difference| per cloth             3.1e-3 / 6.7e-3                 1.4e-2
      (max |dpos| 3.2e-2 / 6.0e-2, not asserted)
"""
import numpy as np
import pytest

from conftest import load_golden

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle.oracle import OracleCloth, params_from_cfg as oracle_params  # noqa: E402  (checker only)

F64 = torch.float64


def _params(W=25, thickness=None, relax=1, reduce_factor=None):
    from gym_cloth_b200 import lib as L
    P = L.default_params()
    P.num_width_points = W; P.num_height_points = W
    if thickness is not None:
        P.thickness = thickness
    if reduce_factor is not None:
        P.reduce_factor = reduce_factor
    P.reserved0 = relax
    OP = oracle_params(None)
    OP.num_width_points = W; OP.num_height_points = W
    OP.thickness = P.thickness; OP.reduce_factor = P.reduce_factor
    OP.ks = P.ks; OP.gravity = P.gravity
    return P, OP


def _bc(P, n, dtype=F64):
    from gym_cloth_b200 import lib as L
    from gym_cloth_b200.batched import BatchedCloth
    return BatchedCloth(P, n, dtype=dtype, mode=L.MODE_COLOURED)


def _oracle(OP, relax, **kw):
    return OracleCloth(OP, mode="coloured", relax_iters=relax, **kw)


def _assert_same(bc, e, o, what=""):
    pos, prev, pin, _ = bc.get_state(e)
    op, oq, opin = o.get_state()
    assert np.array_equal(pos, op), (what, e, np.abs(pos - op).max())
    assert np.array_equal(prev, oq), (what, e, np.abs(prev - oq).max())
    assert np.array_equal(pin, opin.astype(bool)), (what, e)


def _dmax(bc, e, o):
    return np.abs(bc.get_state(e)[0] - o.get_state()[0]).max()


def _grab_set(o, action):
    """The grip list after the oracle's next grab (its release empties o.grabbed by the end of the action); a torn
    cloth is never released, so its old grip stays in the list, as in the kernel's grab count and mask."""
    k = _oracle(o.P, 1)
    k.set_state(*o.get_state(), grabbed=o.grabbed)
    plan = o.decode(action)
    k.grab_top(plan.gx, plan.gy)
    return k.grabbed.tolist()


def _aimed(rng, pos):
    """bench.py's touch_cloth actions: raw U[-1,1]^4 with the grip aimed at a random mesh point of each cloth."""
    a = rng.uniform(-1, 1, size=(len(pos), 4))
    pick = rng.randint(0, pos.shape[1], size=len(pos))
    a[:, :2] = (pos[np.arange(len(pos)), pick, :2] - 0.5) * 2
    return a


# ---------------------------------------------------------------------------------------------- f64, bit for bit
@pytest.mark.parametrize("relax", [1, 2, 3])
def test_f64_one_update_from_phases(relax):
    g = load_golden("phases.npz")
    P, OP = _params(relax=relax)
    bc = _bc(P, 1); o = _oracle(OP, relax)
    bc.set_state(g["pos_0"], g["prev_0"], g["pin_0"], grabbed=g["grabbed"])
    o.set_state(g["pos_0"], g["prev_0"], g["pin_0"], grabbed=g["grabbed"])
    bc.adjust(0.0016, -0.0012, 0.0); o.adjust(0.0016, -0.0012, 0.0)
    bc.update(1); o.update(1)
    torch.cuda.synchronize()
    c = o.counters()
    assert c["collide_hits"] > 0 and c["stretched"] > 0          # both parallel phases have work
    _assert_same(bc, 0, o)
    assert bc.flags.cpu().tolist() == [0]


@pytest.mark.parametrize("relax", [1, 2])
def test_f64_lift_appendix_d(relax):
    g = load_golden("kat_appendix_d.npz")
    P, OP = _params(relax=relax)
    bc = _bc(P, 1); o = _oracle(OP, relax)
    bc.grab_top((0.5, 0.5)); o.grab_top(0.5, 0.5)
    assert bc.grabbed_set(0).tolist() == sorted(o.grabbed.tolist()) == g["grabbed"].tolist()
    for i in range(1, 51):
        bc.adjust(0, 0, 0.0025); o.adjust(0, 0, 0.0025)
        bc.update(1); o.update(1)
        if i in (1, 50):
            _assert_same(bc, 0, o, i)
    assert o.counters()["stretched"] > 0


def _reward(ngrab, cov, prev_cov):
    rew = 0.0
    if ngrab == 0:
        rew += -0.01
    if cov > 0.92:
        rew += 5.
    rew += 0.0
    rew += cov - prev_cov
    return rew


def _actions_vs_oracle(bc, oracles, acts, prev_cov):
    """One step_host action on every env of bc and every oracle; every output must agree."""
    from gym_cloth_b200 import lib as L
    n = len(oracles)
    out = {"sim_steps": np.zeros(n, np.int32), "coverage": np.zeros(n), "flags": np.zeros(n, np.int32),
           "reward": np.zeros(n)}
    bc.step_host(acts, out)
    torch.cuda.synchronize()
    for e, o in enumerate(oracles):
        grabbed = _grab_set(o, acts[e])
        try:
            nupd, ng, _ = o.step_action(acts[e])
        except ZeroDivisionError:
            assert out["flags"][e] & L.FLAG_BADSTATE, e
            continue
        assert out["sim_steps"][e] == nupd, (e, out["sim_steps"][e], nupd)
        assert bc.n_grabbed[e].item() == ng == len(grabbed)
        assert bc.grabbed_set(e).tolist() == sorted(set(grabbed)), e
        flags = (L.FLAG_TEAR if o.tear else 0) | (L.FLAG_OOB if o.out_of_bounds() else 0) | (L.FLAG_NOGRAB if ng == 0 else 0)
        assert out["flags"][e] == flags, (e, out["flags"][e], flags)
        _assert_same(bc, e, o, "action")
        cov = o.coverage()
        assert abs(out["coverage"][e] - cov) <= 1e-12
        assert abs(out["reward"][e] - _reward(ng, cov, prev_cov[e])) <= 1e-12
    return out


@pytest.mark.parametrize("relax", [1, 2, 3])
def test_f64_whole_actions_from_pool(relax):
    """16 crumpled tier-1 reset states, two aimed actions each, through the host entry point (exact decode)."""
    pool = load_golden("bench_pool_t1.npz")
    n = 16
    P, OP = _params(relax=relax)
    bc = _bc(P, n)
    oracles = [_oracle(OP, relax) for _ in range(n)]
    for e in range(n):
        bc.set_state(pool["pos"][e], pool["prev"][e], env=e)
        oracles[e].set_state(pool["pos"][e], pool["prev"][e], np.zeros(625, np.uint8))
    prev_cov = pool["start_coverage"][:n].copy()
    bc.prev_coverage.copy_(torch.from_numpy(prev_cov))
    rng = np.random.RandomState(100 + relax)
    out = _actions_vs_oracle(bc, oracles, _aimed(rng, pool["pos"][:n]), prev_cov)
    assert (out["sim_steps"] > 1400).sum() >= n // 2
    pos = np.stack([o.get_state()[0] for o in oracles])
    _actions_vs_oracle(bc, oracles, _aimed(rng, pos), out["coverage"].copy())


def test_f64_crowded_buckets():
    """45 to 200 points piled into one hash cell (the Jacobi sums over the whole bucket), three updates."""
    rng = np.random.RandomState(11)
    r, c = np.meshgrid(np.arange(25), np.arange(25), indexing="ij")
    flat = np.stack([r / 24.0, c / 24.0, np.zeros_like(r, float)], -1).reshape(-1, 3)
    states = []
    for crowd in (45, 60, 100, 128, 200):
        p = flat.copy()
        idx = rng.choice(625, crowd, replace=False)
        p[idx] = np.array([0.40, 0.40, 0.02]) + rng.uniform(0.0, 1.0, size=(crowd, 3)) * np.array([0.09, 0.09, 0.07])
        states.append(p)
    for relax in (1, 2):
        P, OP = _params(relax=relax)
        bc = _bc(P, len(states))
        for e, p in enumerate(states):
            bc.set_state(p, p, env=e)
        bc.update(3)
        torch.cuda.synchronize()
        for e, p in enumerate(states):
            o = _oracle(OP, relax)
            o.set_state(p, p, np.zeros(625, np.uint8))
            o.update(3)
            assert o.counters()["collide_hits"] > 0
            _assert_same(bc, e, o, ("crowd", relax))


def test_f64_tear_ends_the_action_on_the_oracles_substep():
    from gym_cloth_b200 import lib as L
    g = load_golden("tear.npz")
    P, OP = _params(reduce_factor=float(g["reduce_factor"]))
    n = 2
    acts = np.tile(g["action"][None, :], (n, 1)); acts[1, :2] *= -1.0; acts[1, 2:] *= -0.5
    bc = _bc(P, n)
    oracles = [_oracle(OP, 1) for _ in range(n)]
    out = _actions_vs_oracle(bc, oracles, acts, np.zeros(n))
    assert out["flags"][0] & L.FLAG_TEAR and oracles[0].tear
    assert out["sim_steps"][0] < 1400
    # the torn cloth's next action is a single update
    out2 = _actions_vs_oracle(bc, oracles, acts, out["coverage"].copy())
    assert out2["sim_steps"][0] == 1


def test_f64_badstate_from_hooke_and_from_the_jacobi_collision():
    from gym_cloth_b200 import lib as L
    # coincident connected points: Hooke's l == 0
    P, OP = _params()
    o = _oracle(OP, 1)
    pos, prev, pin = o.get_state()
    pos[1] = pos[0]; prev[1] = prev[0]
    bc = _bc(P, 1)
    bc.set_state(pos, prev, pin)
    o.set_state(pos, prev, pin)
    bc.update(1)
    torch.cuda.synchronize()
    assert bc.flags[0].item() & L.FLAG_BADSTATE
    with pytest.raises(ZeroDivisionError):
        o.update(1)
    # coincident points that share no spring, in one bucket.  Without springs and gravity a resting cloth does not
    # move in Verlet, so the two points are still coincident when the Jacobi collision reads the snapshot.
    P, OP = _params()
    P.ks = 0.0; P.gravity = 0.0; OP.ks = 0.0; OP.gravity = 0.0
    o = _oracle(OP, 1)
    pos, prev, pin = o.get_state()
    pos[300] = pos[20] = (0.3, 0.3, 0.05); prev[:] = pos
    bc = _bc(P, 1)
    bc.set_state(pos, prev, pin)
    o.set_state(pos, prev, pin)
    o.phase("gravity"); o.phase("hookes"); o.phase("verlet"); o.phase("build_map")   # Hooke and Verlet pass
    with pytest.raises(ZeroDivisionError):
        o.phase("self_collide_jacobi")
    o.set_state(pos, prev, pin)
    with pytest.raises(ZeroDivisionError):
        o.update(1)
    bc.update(1)
    torch.cuda.synchronize()
    assert bc.flags[0].item() & L.FLAG_BADSTATE


def test_f64_per_environment_rest_lengths():
    """Three tier-2 cloths with different noise, hence different rest tables, installed per environment."""
    P, OP = _params()
    rng = np.random.RandomState(5)
    n = 3
    bc = _bc(P, n)
    oracles, rests = [], []
    for e in range(n):
        noise = rng.rand(625) * 0.01 - 0.005
        o = _oracle(OP, 1, init_type="tier2", noise=noise, init_side=bool(e % 2))
        rests.append(o.springs()[3])
        pos, prev, pin = o.get_state()
        bc.set_state(pos, prev, pin, env=e)
        bc.set_rest(rests[-1], env=e)
        oracles.append(o)
    assert bc.rest_env_stride == 6 * 625
    assert not np.array_equal(rests[0], rests[1]) and not np.array_equal(rests[1], rests[2])
    bc.update(20)
    for o in oracles:
        o.update(20)
    torch.cuda.synchronize()
    for e, o in enumerate(oracles):
        _assert_same(bc, e, o, "rest")
    pos = np.stack([o.get_state()[0] for o in oracles])
    covs = np.array([o.coverage() for o in oracles])
    bc.prev_coverage.copy_(torch.from_numpy(covs))
    _actions_vs_oracle(bc, oracles, _aimed(rng, pos), covs)


# ---------------------------------------------------------------------------------------------- f32, bounded
TOL_PH = {1: 2.4e-7, 10: 1.3e-6, 50: 1.1e-5}
TOL_AD = {1: 4e-8, 10: 3.6e-7, 50: 3.4e-6}
TOL_POOL = 2.7e-3
TOL_64D = 7.4e-7
TOL_64A = 1.4e-2


def _check(tol, d, what):
    print("%s: %.3e (bound %.1e)" % (what, d, tol))
    assert d <= tol, (what, d, tol)


def test_f32_25x25_substeps():
    g = load_golden("phases.npz")
    P, OP = _params()
    oa = _oracle(OP, 1); ob = _oracle(OP, 1)
    oa.set_state(g["pos_0"], g["prev_0"], g["pin_0"], grabbed=g["grabbed"])
    ph = _bc(P, 1, torch.float32); ad = _bc(P, 1, torch.float32)
    ph.set_state(g["pos_0"], g["prev_0"], g["pin_0"], grabbed=g["grabbed"])
    ad.grab_top((0.5, 0.5)); ob.grab_top(0.5, 0.5)
    assert ad.grabbed_set(0).tolist() == sorted(ob.grabbed.tolist())
    for i in range(1, 51):
        ph.adjust(0.0016, -0.0012, 0.0); oa.adjust(0.0016, -0.0012, 0.0)
        ad.adjust(0, 0, 0.0025); ob.adjust(0, 0, 0.0025)
        ph.update(1); oa.update(1); ad.update(1); ob.update(1)
        if i in TOL_PH:
            torch.cuda.synchronize()
            _check(TOL_PH[i], _dmax(ph, 0, oa), "f32 25x25 phases substep %d" % i)
            _check(TOL_AD[i], _dmax(ad, 0, ob), "f32 25x25 appendix-D substep %d" % i)
    assert np.array_equal(ph.get_state(0)[2], oa.get_state()[2].astype(bool))


def test_f32_25x25_pool_actions():
    pool = load_golden("bench_pool_t1.npz")
    n = 64
    P, OP = _params()
    bc = _bc(P, n, torch.float32)
    for e in range(n):
        bc.set_state(pool["pos"][e], pool["prev"][e], env=e)
    acts = _aimed(np.random.RandomState(7), pool["pos"])
    out = {"sim_steps": np.zeros(n, np.int32), "coverage": np.zeros(n)}
    bc.step_host(acts, out)
    torch.cuda.synchronize()
    covs, dmax = np.zeros(n), 0.0
    for e in range(n):
        o = _oracle(OP, 1)
        o.set_state(pool["pos"][e], pool["prev"][e], np.zeros(625, np.uint8))
        grabbed = _grab_set(o, acts[e])
        nupd, ng, _ = o.step_action(acts[e])
        assert out["sim_steps"][e] == nupd, e
        assert bc.grabbed_set(e).tolist() == sorted(set(grabbed)), e
        covs[e] = o.coverage()
        dmax = max(dmax, _dmax(bc, e, o))
    print("f32 25x25 pool max |dpos| %.3e, max |dcov| %.3e" % (dmax, np.abs(out["coverage"] - covs).max()))
    _check(TOL_POOL, abs(out["coverage"].mean() - covs.mean()), "f32 25x25 pool |d mean coverage|")


def _drive(bc, o):
    bc.grab_top((0.5, 0.5)); o.grab_top(0.5, 0.5)
    assert bc.n_grabbed[0].item() == len(o.grabbed) > 0
    for i in range(12):
        bc.adjust(0.0, 0.0, 0.0025); o.adjust(0.0, 0.0, 0.0025)
        bc.update(1); o.update(1)
    for i in range(6):
        bc.adjust(0.002, -0.001, 0.0); o.adjust(0.002, -0.001, 0.0)
        bc.update(1); o.update(1)


@pytest.mark.parametrize("relax", [1, 2])
def test_f32_64x64_config4(relax):
    """BASELINE config 4: 64x64 cloths, thickness 0.006 (2*thickness below the grid spacing)."""
    P, OP = _params(W=64, thickness=0.006, relax=relax)
    bc = _bc(P, 1, torch.float32); o = _oracle(OP, relax)
    assert o.N == 4096
    _drive(bc, o)
    torch.cuda.synchronize()
    _check(TOL_64D, _dmax(bc, 0, o), "f32 64x64 relax %d drive" % relax)
    assert np.array_equal(bc.get_state(0)[2], o.get_state()[2].astype(bool))
    acts = np.array([[0.0, 0.0, 0.3, 0.1], [0.5, 0.5, -0.2, 0.2], [-0.4, 0.3, 0.1, -0.3]])
    n = len(acts)
    bc = _bc(P, n, torch.float32)
    out = {"sim_steps": np.zeros(n, np.int32), "coverage": np.zeros(n), "flags": np.zeros(n, np.int32)}
    bc.step_host(acts, out)
    torch.cuda.synchronize()
    for e in range(n):
        o = _oracle(OP, relax)
        grabbed = _grab_set(o, acts[e])
        nupd, ng, _ = o.step_action(acts[e])
        assert out["sim_steps"][e] == nupd and bc.n_grabbed[e].item() == ng > 0, e
        assert bc.grabbed_set(e).tolist() == sorted(set(grabbed)), e
        assert not (out["flags"][e] & 8) and bool(out["flags"][e] & 1) == o.tear
        print("f32 64x64 relax %d action env %d max |dpos| %.3e" % (relax, e, _dmax(bc, e, o)))
        _check(TOL_64A, abs(out["coverage"][e] - o.coverage()), "f32 64x64 relax %d action |dcov|" % relax)
