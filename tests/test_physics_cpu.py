"""Per-environment material without a GPU: the ClothB200Physics layout, the `_phys` entry points' argument checks and
BatchedClothEnv's host-side validation of set_physics / get_physics."""
import ctypes as C
import os

import numpy as np
import pytest

from gym_cloth_b200 import lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sizeof_physics_matches_ctypes():
    assert L.lib().clothb200_sizeof_physics() == C.sizeof(L.Physics) == 64
    assert [f for f, _ in L.Physics._fields_][:6] == list(L.PHYSICS_FIELDS)


def test_phys_symbols_exported_and_declared():
    lib = L.lib()
    with open(os.path.join(ROOT, "include", "clothb200.h")) as fh:
        header = fh.read()
    names = ["clothb200_sizeof_physics"] + ["clothb200_%s_phys_%s" % (b, s) for b in ("step_plans", "step_actions", "update_n", "step_host")
                                            for s in ("f32", "f64")]
    for n in names:
        assert hasattr(lib, n), n
        assert n + "(" in header, n
        assert n in L.exported_symbols(), n


def test_phys_argument_errors_without_gpu():
    """Argument errors are found before anything touches a device: -1 (CLOTHB200_ERR_ARG)."""
    lib = L.lib()
    P = L.default_params()
    io = L.Step()
    rows = (L.Physics * 2)()
    for sfx in ("_f32", "_f64"):
        assert getattr(lib, "clothb200_step_plans_phys" + sfx)(C.byref(P), 0, -1, None, C.byref(io), 0, rows, None) == -1
        assert getattr(lib, "clothb200_step_plans_phys" + sfx)(C.byref(P), 0, 2, None, None, 0, rows, None) == -1
        assert getattr(lib, "clothb200_update_n_phys" + sfx)(C.byref(P), 0, 2, -1, C.byref(io), rows, None) == -1
        assert getattr(lib, "clothb200_update_n_phys" + sfx)(C.byref(P), 0, -3, 1, C.byref(io), rows, None) == -1
        assert getattr(lib, "clothb200_step_actions_phys" + sfx)(C.byref(P), 0, 2, None, None, C.byref(io), 0, rows, None) == -1
        assert getattr(lib, "clothb200_step_host_phys" + sfx)(None, 0, 2, None, C.byref(io), 0, *([None] * 7), rows, None) == -1
        # n_env == 0 is a no-op, as for the plain entry points
        assert getattr(lib, "clothb200_update_n_phys" + sfx)(C.byref(P), 0, 0, 1, C.byref(io), rows, None) == 0


class _NoGpuEnv(object):
    """BatchedClothEnv's physics methods on a stand-in batch: they validate on the host before touching the device."""

    def __init__(self, n_env):
        from gym_cloth_b200.envs.cloth_env import BatchedClothEnv, load_cfg
        from gym_cloth_b200 import cfg_path
        self.env = BatchedClothEnv.__new__(BatchedClothEnv)
        self.env.cfg = load_cfg(cfg_path(1))
        self.env.P = L.params_from_cfg(self.env.cfg)
        self.env.n_env = n_env
        self.calls = []
        outer = self

        class _Cloth(object):
            physics = None

            def set_physics(self, envs=None, **fields):
                outer.calls.append((None if envs is None else np.asarray(envs).tolist(), fields))
        self.env.cloth = _Cloth()


def test_get_physics_defaults_to_cfg():
    e = _NoGpuEnv(3).env
    ph = e.get_physics()
    assert sorted(ph) == sorted(L.PHYSICS_FIELDS)
    cl = e.cfg["cloth"]
    for k in ("density", "ks", "damping", "plane_friction", "tear_thresh"):
        assert ph[k].tolist() == [float(cl[k])] * 3, k
    assert ph["gravity"].tolist() == [-9.8] * 3


@pytest.mark.parametrize("field", list(L.PHYSICS_FIELDS))
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_set_physics_rejects_non_finite(field, bad):
    h = _NoGpuEnv(3)
    with pytest.raises(ValueError):
        h.env.set_physics(**{field: bad})
    with pytest.raises(ValueError):
        h.env.set_physics(envs=[0, 2], **{field: [1.0, bad]})
    assert h.calls == []


@pytest.mark.parametrize("density", [0.0, -1.0, [200.0, 0.0]])
def test_set_physics_rejects_non_positive_density(density):
    h = _NoGpuEnv(2)
    with pytest.raises(ValueError):
        h.env.set_physics(density=density)
    assert h.calls == []


def test_set_physics_rejects_wrong_length():
    h = _NoGpuEnv(4)
    with pytest.raises(ValueError):
        h.env.set_physics(ks=[1.0, 2.0, 3.0])
    with pytest.raises(ValueError):
        h.env.set_physics(envs=[1, 2], damping=[1.0, 2.0, 3.0])
    with pytest.raises(ValueError):
        h.env.set_physics(envs=[1, 2], damping=np.ones((2, 1)))
    with pytest.raises(ValueError):
        h.env.set_physics(envs=[5], damping=1.0)
    assert h.calls == []


def test_set_physics_passes_valid_values():
    h = _NoGpuEnv(4)
    h.env.set_physics(envs=[1, 3], density=[100.0, 300.0], gravity=-7.5)
    (envs, fields), = h.calls
    assert envs == [1, 3]
    assert fields["density"].tolist() == [100.0, 300.0] and fields["gravity"].tolist() == [-7.5, -7.5]
    assert set(fields) == {"density", "gravity"}
