"""Time-sliced step (ClothB200Step.sched_scratch_bytes): a persistent grid runs a few substeps of a cloth, parks it and
takes the next one.  Results must not depend on it: f64 bit for bit, and every output (grip, substeps, flags, reward)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def queue_parks(c):
    """Cloths parked by the last sliced launch of BatchedCloth c: the queue counters are the last 16 bytes of
    sched_scratch (cloth_abi.cu, clothb200_sched_scratch_bytes); tickets issued = n_env + one per park."""
    qctl = c.sched_scratch[-16:].cpu().numpy().view(np.int32)
    return int(qctl[1]) - c.n_env


def _run(dtype, n, sliced, actions, slots=3, q=37, tier=1, parks=None):
    """q = 0 keeps the production slice length, swap hysteresis and endgame (CLOTHB200_SLICE and friends)."""
    from gym_cloth_b200 import cfg_path, lib as L
    from gym_cloth_b200.envs import BatchedClothEnv
    lib = L.lib()
    lib.clothb200_debug_set_slicing(0, 0)
    env = BatchedClothEnv(cfg_path(tier), n, dtype=dtype, seed=21)
    env.reset()                                  # resets step subsets through env_order: never sliced
    env.cloth.time_slice = sliced
    if sliced:
        lib.clothb200_debug_set_slicing(slots, q)
    outs = []
    try:
        for a in actions:
            obs, rew, done, info = env.step(torch.from_numpy(a).to(env.device, env.torch_dtype))
            c = env.cloth
            if parks is not None:
                parks.append(queue_parks(c))
            outs.append({k: v.clone().cpu().numpy() for k, v in dict(pos=c.pos, prev=c.prev, rew=rew, done=done, sim=c.sim_steps, ngrab=c.n_grabbed,
                                                                       flags=c.flags, cov=c.coverage, nss=c.num_sim_steps, mask=c.grab_mask).items()})
    finally:
        lib.clothb200_debug_set_slicing(0, 0)
    return outs


def _actions(n, k, seed=4):
    rng = np.random.RandomState(seed)
    a = [rng.uniform(-1, 1, size=(n, 4)) for _ in range(k)]
    for x in a:
        x[:, :2] *= 0.85                          # mostly on the cloth, some misses stay (0 substeps)
    return a


def test_sliced_f64_is_bit_identical():
    n = 10
    acts = _actions(n, 2)
    ref = _run("f64", n, False, acts)
    for slots, q in ((3, 37), (7, 500), (1, 211)):
        got = _run("f64", n, True, acts, slots=slots, q=q)
        for r, g in zip(ref, got):
            for k in r:
                assert np.array_equal(r[k], g[k]), (slots, q, k)
    assert (ref[0]["sim"] > 0).any() and (ref[0]["sim"] == 0).any()


def test_sliced_f32_matches_unsliced():
    n = 24
    acts = _actions(n, 2, seed=9)
    ref = _run("f32", n, False, acts)
    got = _run("f32", n, True, acts, slots=5, q=64)
    again = _run("f32", n, True, acts, slots=5, q=64)
    for r, g, h in zip(ref, got, again):
        for k in r:
            assert np.array_equal(g[k], h[k]), k          # deterministic
        for k in ("sim", "ngrab", "mask", "done"):
            assert np.array_equal(r[k], g[k]), k
        assert np.array_equal(r["pos"], g["pos"]) and np.array_equal(r["rew"], g["rew"])
    # queue stress: two-substep slices on four slots = ~20 000 swaps through a 24-slot ring
    hammer = _run("f32", n, True, acts[:1], slots=4, q=2)
    assert np.array_equal(ref[0]["pos"], hammer[0]["pos"]) and np.array_equal(ref[0]["sim"], hammer[0]["sim"])


def test_sliced_tear_and_tier2_rest_lengths():
    from gym_cloth_b200 import lib as L
    from gym_cloth_b200.batched import BatchedCloth
    lib = L.lib()
    # a violent pull (the tear fixture's reduce_factor and action) tears the cloth mid-slice: the action ends there, in
    # the same substep as unsliced, and the torn cloth's next action is a single update
    from conftest import load_golden
    g = load_golden("tear.npz")
    P = L.default_params(); P.reduce_factor = float(g["reduce_factor"])
    res = []
    for sliced in (False, True):
        bc = BatchedCloth(P, 6, dtype=torch.float64)
        bc.time_slice = sliced
        a = np.tile(g["action"][None, :], (6, 1)); a[3:, :2] *= -1.0; a[3:, 2:] *= -0.5
        if sliced:
            lib.clothb200_debug_set_slicing(2, 50)
        try:
            bc.step_actions(torch.from_numpy(a).cuda())
            first = (bc.pos.clone(), bc.sim_steps.clone(), bc.flags.clone())
            bc.step_actions(torch.from_numpy(a).cuda())
            res.append(first + (bc.pos.clone(), bc.sim_steps.clone(), bc.flags.clone()))
        finally:
            lib.clothb200_debug_set_slicing(0, 0)
    for x, y in zip(res[0], res[1]):
        assert torch.equal(x, y)
    assert ((res[0][2] & 1) != 0).any() and int(res[0][1][0]) == int(g["info"][1]) and int(res[0][4][0]) == 1
    acts = _actions(6, 1, seed=2)
    ref = _run("f64", 6, False, acts, tier=2)
    got = _run("f64", 6, True, acts, slots=2, q=100, tier=2)
    for k in ref[0]:
        assert np.array_equal(ref[0][k], got[0][k]), k


def test_crowded_buckets_replay_from_registers_bit_exact():
    """Crumpled cloths pile 40-100+ points into one hash cell; buckets of 33-64 and 65-128 members are replayed out of
    registers (two / four members per lane), larger ones from shared memory.  All must equal the sequential oracle."""
    from gym_cloth_b200 import lib as L
    from gym_cloth_b200.batched import BatchedCloth
    from oracle.oracle import OracleCloth
    rng = np.random.RandomState(11)
    r, c = np.meshgrid(np.arange(25), np.arange(25), indexing="ij")
    flat = np.stack([r / 24.0, c / 24.0, np.zeros_like(r, float)], -1).reshape(-1, 3)
    states = []
    for crowd in (45, 60, 100, 128, 200):
        p = flat.copy()
        idx = rng.choice(625, crowd, replace=False)
        # the chosen points are squeezed into one 0.125 cell, a few layers thick
        p[idx] = np.array([0.40, 0.40, 0.02]) + rng.uniform(0.0, 1.0, size=(crowd, 3)) * np.array([0.09, 0.09, 0.07])
        states.append(p)
    n = len(states)
    bc = BatchedCloth(L.default_params(), n, dtype=torch.float64)
    for e, p in enumerate(states):
        bc.set_state(p, p, env=e)
    bc.update(3)
    torch.cuda.synchronize()
    for e, p in enumerate(states):
        o = OracleCloth()
        o.set_state(p, p, np.zeros(625, np.uint8))
        o.update(3)
        pos, prev, _, _ = bc.get_state(e)
        op, oq, _ = o.get_state()
        assert np.array_equal(pos, op) and np.array_equal(prev, oq), (e, np.abs(pos - op).max())
    # f32 build: same states within the single-update tolerance scale (3 updates of a violent state)
    b32 = BatchedCloth(L.default_params(), n, dtype=torch.float32)
    for e, p in enumerate(states):
        b32.set_state(p, p, env=e)
    b32.update(3)
    d = (b32.pos.double() - bc.pos)[:, :, :3].abs().amax().item()
    assert d < 2e-4, d
