"""Time slicing with the production schedule: slice 64 substeps, swap hysteresis 128, quarter slices for the last 12
slices of an action (cloth_kernels.cuh).  clothb200_debug_set_slicing(slots, 0) only forces a small slot count, so
cloths are parked and resumed under the same knobs a full launch uses.  Every output must equal the unsliced run
(time_slice = False: one CTA per cloth for a whole action), bit for bit in f32 too, since a resumed cloth replays the
same substeps.  Each case also reads the queue counters to show that cloths were in fact parked."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import load_golden
from test_gpu_slicing import _actions, _run, queue_parks

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("pos", "prev", "reward", "done", "sim_steps", "n_grabbed", "flags", "coverage", "num_sim_steps", "grab_mask")


def _compare(ref, got, what):
    for r, g in zip(ref, got):
        for k in r:
            assert np.array_equal(r[k], g[k]), (what, k)


@pytest.mark.parametrize("dtype,n,slots,tier,seed", [("f64", 10, 3, 1, 4), ("f32", 24, 5, 1, 9), ("f64", 6, 2, 2, 2)])
def test_reference_order_production_slicing(dtype, n, slots, tier, seed):
    acts = _actions(n, 2, seed=seed)
    ref = _run(dtype, n, False, acts, tier=tier)
    parks = []
    got = _run(dtype, n, True, acts, slots=slots, q=0, tier=tier, parks=parks)
    _compare(ref, got, (dtype, tier))
    assert len(set(int(x) for x in ref[0]["sim"][ref[0]["sim"] > 0])) > 1      # varied iters_pull
    assert sum(parks) > 0, parks


def _coloured(dtype, W, n, relax, actions, sliced, slots=0, q=0, thickness=None):
    from gym_cloth_b200 import lib as L
    from gym_cloth_b200.batched import BatchedCloth
    lib = L.lib()
    P = L.default_params()
    P.num_width_points = W; P.num_height_points = W; P.reserved0 = relax
    if thickness is not None:
        P.thickness = thickness
    tdt = torch.float64 if dtype == "f64" else torch.float32
    bc = BatchedCloth(P, n, dtype=tdt, mode=L.MODE_COLOURED)
    if W == 25:
        pool = load_golden("bench_pool_t1.npz")
        for e in range(n):
            bc.set_state(pool["pos"][e], pool["prev"][e], env=e)
    bc.time_slice = sliced
    outs, parks = [], []
    lib.clothb200_debug_set_slicing(slots if sliced else 0, q if sliced else 0)
    try:
        for a in actions:
            bc.step_actions(torch.from_numpy(a).to(bc.device, tdt))
            torch.cuda.synchronize()
            parks.append(queue_parks(bc))
            outs.append({k: getattr(bc, k).clone().cpu().numpy() for k in KEYS})
    finally:
        lib.clothb200_debug_set_slicing(0, 0)
    return outs, parks


@pytest.mark.parametrize("dtype,W,n,slots,relax,thickness", [("f64", 25, 8, 3, 1, None), ("f32", 64, 6, 2, 2, 0.006)])
def test_coloured_production_slicing(dtype, W, n, slots, relax, thickness):
    acts = _actions(n, 2, seed=13)
    for a in acts:
        a[:, :2] *= 0.6                                             # mostly on the cloth
    ref, _ = _coloured(dtype, W, n, relax, acts, False, thickness=thickness)
    got, parks = _coloured(dtype, W, n, relax, acts, True, slots=slots, thickness=thickness)
    _compare(ref, got, (dtype, W))
    assert sum(parks) > 0, parks
    assert len(set(ref[0]["sim_steps"].tolist())) > 1


def test_coloured_two_substep_hammer():
    acts = _actions(8, 1, seed=3)
    ref, _ = _coloured("f64", 25, 8, 1, acts, False)
    got, parks = _coloured("f64", 25, 8, 1, acts, True, slots=4, q=2)
    _compare(ref, got, "hammer")
    assert parks[0] > 100, parks


# The knobs are read once per process: this case runs in a child process with slices of one substep (CLOTHB200_SLICE=7
# shifted right by 3 in the endgame, which here is the whole action) and no hysteresis.  Every substep ends a slice, and
# with equal actions most of them end in a swap (about 8 000 parks over 12 600 substep boundaries per action on a B200),
# so cloths are also resumed exactly at the substep that releases the gripper.
CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from test_gpu_slicing import _run
acts = [np.load(sys.argv[2])[i] for i in range(2)]
parks = []
outs = _run("f64", 8, True, acts, slots=3, q=0, parks=parks)
np.savez(sys.argv[3], parks=np.array(parks), **{"%d_%s" % (i, k): v for i, o in enumerate(outs) for k, v in o.items()})
"""


def test_knob_environment_variables_in_a_child_process(tmp_path):
    n = 8
    acts = _actions(n, 2, seed=21)
    for a in acts:
        a[:, :2] *= 0.5
        a[:, 2:] = (0.29, 0.04)                                     # one pull length: equal actions, parks everywhere
    np.save(tmp_path / "acts.npy", np.stack(acts))
    env = dict(os.environ, CLOTHB200_SLICE="7", CLOTHB200_YIELD_SLACK="0", CLOTHB200_ENDGAME="1000",
               CLOTHB200_ENDGAME_SHIFT="3")
    out = tmp_path / "child.npz"
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(tmp_path / "acts.npy"), str(out)], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-4000:]
    ref = _run("f64", n, False, acts)
    got = np.load(out)
    for i, o in enumerate(ref):
        for k in o:
            assert np.array_equal(o[k], got["%d_%s" % (i, k)]), (i, k)
    sims = ref[0]["sim"]
    assert (sims > 1400).sum() > 3
    print("child: parks per action %s, substeps %s" % (got["parks"].tolist(), sims.tolist()))
    assert got["parks"][0] >= int(np.maximum(sims - 1, 0).sum()) // 4, (got["parks"], sims)
