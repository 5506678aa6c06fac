"""ctypes wrapper around oracle/liboracle.so (TEST INFRASTRUCTURE, never imported by
gym_cloth_b200/).  See cloth_oracle.c for the reference citations of every function.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline / `--impl reference`
legs may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liboracle.so")


class OracleParams(C.Structure):
    _fields_ = [
        ("num_width_points", C.c_int32), ("num_height_points", C.c_int32),
        ("width", C.c_double), ("height", C.c_double),
        ("density", C.c_double), ("ks", C.c_double), ("damping", C.c_double),
        ("thickness", C.c_double), ("plane_friction", C.c_double), ("tear_thresh", C.c_double),
        ("gravity", C.c_double), ("minimum_z", C.c_double),
        ("frames_per_sec", C.c_int32), ("simulation_steps", C.c_int32),
        ("iters_up", C.c_double), ("iters_up_rest", C.c_double),
        ("iters_grip_rest", C.c_double), ("iters_rest", C.c_double),
        ("iters_pull_max", C.c_int32),
        ("reduce_factor", C.c_double), ("grip_radius", C.c_double), ("gripper_height", C.c_double),
        ("clip_act_space", C.c_int32), ("delta_actions", C.c_int32), ("max_actions", C.c_int32),
        ("pad_", C.c_int32),
    ]


class OraclePlan(C.Structure):
    _fields_ = [("gx", C.c_double), ("gy", C.c_double), ("dxr", C.c_double), ("dyr", C.c_double),
                ("iters_pull", C.c_int32), ("pad_", C.c_int32)]


_lib = None


def build(force=False):
    src = os.path.join(HERE, "cloth_oracle.c")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", HERE, "-B", "liboracle.so"],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(LIB_PATH)
    dp = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
    u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
    i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
    i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
    vp = C.c_void_p
    PP = C.POINTER(OracleParams)
    L.oracle_params_default.argtypes = [PP]
    L.oracle_sizeof_params.restype = C.c_int
    L.oracle_cloth_create.argtypes = [PP, C.c_int, C.c_void_p, C.c_int]
    L.oracle_cloth_create.restype = vp
    L.oracle_cloth_destroy.argtypes = [vp]
    for name in ("num_points", "num_springs", "tear", "num_grabbed"):
        f = getattr(L, "oracle_cloth_" + name); f.argtypes = [vp]; f.restype = C.c_int
    L.oracle_cloth_set_tear.argtypes = [vp, C.c_int]
    L.oracle_cloth_get_grabbed.argtypes = [vp, i32p]
    L.oracle_cloth_set_grabbed.argtypes = [vp, i32p, C.c_int]
    L.oracle_cloth_get_state.argtypes = [vp, dp, dp, u8p]
    L.oracle_cloth_set_state.argtypes = [vp, dp, dp, u8p]
    L.oracle_cloth_get_force.argtypes = [vp, dp]
    L.oracle_cloth_get_springs.argtypes = [vp, i32p, i32p, u8p, dp]
    L.oracle_cloth_set_rest.argtypes = [vp, dp]
    L.oracle_cloth_get_counters.argtypes = [vp, i64p]
    L.oracle_cloth_set_mode.argtypes = [vp, C.c_int, C.c_int]; L.oracle_cloth_set_mode.restype = None
    L.oracle_cloth_get_colours.argtypes = [vp, i32p]; L.oracle_cloth_get_colours.restype = None
    for name in ("gravity", "verlet", "plane", "limit"):
        f = getattr(L, "oracle_phase_" + name); f.argtypes = [vp]; f.restype = None
    for name in ("hookes", "build_map", "self_collide", "self_collide_jacobi"):
        f = getattr(L, "oracle_phase_" + name); f.argtypes = [vp]; f.restype = C.c_int
    L.oracle_phase_limit_coloured.argtypes = [vp, C.c_int]; L.oracle_phase_limit_coloured.restype = None
    L.oracle_update.argtypes = [vp]; L.oracle_update.restype = C.c_int
    L.oracle_update_coloured.argtypes = [vp]; L.oracle_update_coloured.restype = C.c_int
    L.oracle_update_n.argtypes = [vp, C.c_int]; L.oracle_update_n.restype = C.c_int
    L.oracle_grab_top.argtypes = [vp, C.c_double, C.c_double, C.c_double]; L.oracle_grab_top.restype = C.c_int
    L.oracle_grab.argtypes = [vp, C.c_double, C.c_double, C.c_double]; L.oracle_grab.restype = C.c_int
    L.oracle_adjust.argtypes = [vp, C.c_double, C.c_double, C.c_double]; L.oracle_adjust.restype = None
    L.oracle_release.argtypes = [vp]; L.oracle_release.restype = None
    L.oracle_decode_action.argtypes = [PP, dp, C.POINTER(OraclePlan)]
    L.oracle_run_plan.argtypes = [vp, C.POINTER(OraclePlan), C.c_int, C.POINTER(C.c_int)]
    L.oracle_run_plan.restype = C.c_int
    L.oracle_step_action.argtypes = [vp, dp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.oracle_step_action.restype = C.c_int
    L.oracle_hull_area.argtypes = [dp, C.c_int]; L.oracle_hull_area.restype = C.c_double
    L.oracle_coverage.argtypes = [vp]; L.oracle_coverage.restype = C.c_double
    L.oracle_variance_inv.argtypes = [vp]; L.oracle_variance_inv.restype = C.c_double
    L.oracle_out_of_bounds.argtypes = [vp]; L.oracle_out_of_bounds.restype = C.c_int
    assert L.oracle_sizeof_params() == C.sizeof(OracleParams)
    _lib = L
    return L


def params_from_cfg(cfg=None):
    """OracleParams from a gym-cloth cfg dict (the yaml the reference loads at
    cloth_env.py:87-88); defaults = cfg/t1_rgbd.yaml."""
    P = OracleParams()
    lib().oracle_params_default(C.byref(P))
    if cfg is None:
        return P
    cl, env = cfg["cloth"], cfg["env"]
    P.num_width_points = cl["num_width_points"]; P.num_height_points = cl["num_height_points"]
    P.width = cl["width"]; P.height = cl["height"]
    P.density = cl["density"]; P.ks = cl["ks"]; P.damping = cl["damping"]
    P.thickness = cl["thickness"]; P.plane_friction = cl["plane_friction"]
    P.tear_thresh = cl["tear_thresh"]
    P.frames_per_sec = cfg["frames_per_sec"]; P.simulation_steps = cfg["simulation_steps"]
    P.iters_up = env["iters_up"]; P.iters_up_rest = env["iters_up_rest"]
    P.iters_grip_rest = env["iters_grip_rest"]; P.iters_rest = env["iters_rest"]
    P.iters_pull_max = env["iters_pull_max"]
    P.reduce_factor = env["reduce_factor"]; P.grip_radius = env["grip_radius"]
    P.gripper_height = cl["height"]  # Gripper(cloth, grip_radius, cfg.cloth.height, ...) cloth_env.py:752-753
    P.clip_act_space = int(bool(env["clip_act_space"])); P.delta_actions = int(bool(env["delta_actions"]))
    P.max_actions = env["max_actions"]
    return P


_TIER = {"tier1": 1, "tier2": 2, "tier3": 3, 1: 1, 2: 2, 3: 3}
_MODE = {"reference_order": 0, "coloured": 1}


class OracleCloth(object):
    """One cloth + gripper, the CPU restatement of Cloth/Gripper/ClothEnv.step.

    mode="coloured" makes update() and step_action() run oracle_update_coloured (the specification of the
    graph-coloured kernels, CLOTHB200_MODE_COLOURED) with max(1, relax_iters) limit passes per update."""

    def __init__(self, params=None, init_type="tier1", noise=None, init_side=True, mode="reference_order", relax_iters=1):
        self.L = lib()
        self.P = params if params is not None else params_from_cfg(None)
        nz = None
        if noise is not None:
            nz = np.ascontiguousarray(noise, dtype=np.float64)
        self.h = self.L.oracle_cloth_create(C.byref(self.P), _TIER[init_type],
                                            nz.ctypes.data if nz is not None else None,
                                            int(bool(init_side)))
        if not self.h:
            raise ValueError("oracle_cloth_create failed (non-square grid or bad init type)")
        self.N = self.L.oracle_cloth_num_points(self.h)
        self.S = self.L.oracle_cloth_num_springs(self.h)
        self.mode = mode
        self.L.oracle_cloth_set_mode(self.h, _MODE[mode], int(relax_iters))

    def __del__(self):
        try:
            if self.h:
                self.L.oracle_cloth_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # --- state ---
    def get_state(self):
        pos = np.empty((self.N, 3)); prev = np.empty((self.N, 3)); pin = np.empty(self.N, np.uint8)
        self.L.oracle_cloth_get_state(self.h, pos, prev, pin)
        return pos, prev, pin

    def set_state(self, pos, prev, pinned, grabbed=None, tear=None):
        self.L.oracle_cloth_set_state(self.h, np.ascontiguousarray(pos, np.float64),
                                      np.ascontiguousarray(prev, np.float64),
                                      np.ascontiguousarray(pinned, np.uint8))
        if grabbed is not None:
            g = np.ascontiguousarray(grabbed, np.int32)
            self.L.oracle_cloth_set_grabbed(self.h, g, len(g))
        if tear is not None:
            self.L.oracle_cloth_set_tear(self.h, int(tear))

    @property
    def pos(self):
        return self.get_state()[0]

    @property
    def tear(self):
        return bool(self.L.oracle_cloth_tear(self.h))

    @property
    def grabbed(self):
        n = self.L.oracle_cloth_num_grabbed(self.h)
        out = np.empty(max(n, 1), np.int32)
        self.L.oracle_cloth_get_grabbed(self.h, out)
        return out[:n].copy()

    def force(self):
        f = np.empty((self.N, 3)); self.L.oracle_cloth_get_force(self.h, f); return f

    def springs(self):
        a = np.empty(self.S, np.int32); b = np.empty(self.S, np.int32)
        t = np.empty(self.S, np.uint8); r = np.empty(self.S)
        self.L.oracle_cloth_get_springs(self.h, a, b, t, r)
        return a, b, t, r

    def colours(self):
        """Colour class 2*kind + parity of every spring (coloured mode), in spring-list order."""
        out = np.empty(self.S, np.int32); self.L.oracle_cloth_get_colours(self.h, out); return out

    def set_rest(self, rest):
        self.L.oracle_cloth_set_rest(self.h, np.ascontiguousarray(rest, np.float64))

    def counters(self):
        out = np.zeros(5, np.int64); self.L.oracle_cloth_get_counters(self.h, out)
        return dict(zip(("updates", "pair_tests", "collide_hits", "stretched", "plane"), out.tolist()))

    # --- physics ---
    def _chk(self, rc):
        if rc == -1:
            raise ZeroDivisionError("float division")
        if rc == -2:
            raise ValueError("cannot convert float NaN/inf to integer")
        if rc < 0:
            raise RuntimeError("oracle error %d" % rc)
        return rc

    def phase(self, name, *args):
        r = getattr(self.L, "oracle_phase_" + name)(self.h, *args)
        if r is not None:
            self._chk(r)

    def update(self, n=1):
        self._chk(self.L.oracle_update_n(self.h, int(n)))

    def grab_top(self, x, y, grip_radius=None):
        return self.L.oracle_grab_top(self.h, x, y, self.P.grip_radius if grip_radius is None else grip_radius)

    def grab(self, x, y, grip_radius=None):
        return self.L.oracle_grab(self.h, x, y, self.P.grip_radius if grip_radius is None else grip_radius)

    def adjust(self, x, y, z):
        self.L.oracle_adjust(self.h, x, y, z)

    def release(self):
        self.L.oracle_release(self.h)

    def decode(self, action):
        plan = OraclePlan()
        self.L.oracle_decode_action(C.byref(self.P), np.ascontiguousarray(action, np.float64), C.byref(plan))
        return plan

    def step_action(self, action, force_grab=False):
        """cloth_env.py:401-515.  Returns (num_updates, n_grabbed, iters_pull)."""
        ng = C.c_int(0); ip = C.c_int(0)
        n = self._chk(self.L.oracle_step_action(self.h, np.ascontiguousarray(action, np.float64),
                                                int(force_grab), C.byref(ng), C.byref(ip)))
        return n, ng.value, ip.value

    # --- reward terms ---
    def coverage(self):
        return self.L.oracle_coverage(self.h)

    def variance_inv(self):
        return self.L.oracle_variance_inv(self.h)

    def out_of_bounds(self):
        return bool(self.L.oracle_out_of_bounds(self.h))


def hull_area(xy):
    xy = np.ascontiguousarray(xy, np.float64)
    return lib().oracle_hull_area(xy, len(xy))
