"""ctypes binding of libclothb200.so (the C ABI declared in include/clothb200.h).

There is no CPU fallback: if the shared library has not been built, importing this module's
`lib()` raises.  Build it with `python -m gym_cloth_b200.build` (nvcc, sm_100a).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libclothb200.so")

OK = 0
FLAG_TEAR, FLAG_OOB, FLAG_NOGRAB, FLAG_BADSTATE = 1, 2, 4, 8
MODE_REFERENCE_ORDER, MODE_COLOURED = 0, 1
REWARD_TYPE = {"coverage-delta": 0, "coverage": 1}
INIT_TIER = {"tier1": 1, "tier2": 2, "tier3": 3}


class ClothB200Error(RuntimeError):
    """`code` is the CLOTHB200_ERR_* return code of the failed library call (None when no call failed)."""

    def __init__(self, msg, code=None):
        RuntimeError.__init__(self, msg)
        self.code = code


class Params(C.Structure):
    """ClothB200Params (include/clothb200.h)."""
    _fields_ = [
        ("num_width_points", C.c_int32), ("num_height_points", C.c_int32),
        ("width", C.c_double), ("height", C.c_double),
        ("density", C.c_double), ("ks", C.c_double), ("damping", C.c_double),
        ("thickness", C.c_double), ("plane_friction", C.c_double), ("tear_thresh", C.c_double),
        ("gravity", C.c_double), ("minimum_z", C.c_double),
        ("frames_per_sec", C.c_int32), ("simulation_steps", C.c_int32),
        ("iters_up", C.c_double), ("iters_up_rest", C.c_double),
        ("iters_grip_rest", C.c_double), ("iters_rest", C.c_double),
        ("iters_pull_max", C.c_int32), ("max_actions", C.c_int32),
        ("reduce_factor", C.c_double), ("grip_radius", C.c_double), ("gripper_height", C.c_double),
        ("clip_act_space", C.c_int32), ("delta_actions", C.c_int32),
        ("force_grab", C.c_int32), ("reserved0", C.c_int32),
        ("reward_type", C.c_int32), ("reserved1", C.c_int32),
    ]


class Plan(C.Structure):
    """ClothB200Plan."""
    _fields_ = [("gx", C.c_double), ("gy", C.c_double), ("dxr", C.c_double), ("dyr", C.c_double),
                ("iters_pull", C.c_int32), ("reserved", C.c_int32)]


class Step(C.Structure):
    """ClothB200Step: device pointers of every per-environment tensor."""
    _fields_ = [
        ("pos", C.c_void_p), ("prev", C.c_void_p),
        ("rest", C.c_void_p), ("rest_env_stride", C.c_int64),
        ("flags", C.c_void_p), ("sim_steps", C.c_void_p), ("n_grabbed", C.c_void_p), ("grab_mask", C.c_void_p),
        ("coverage", C.c_void_p), ("variance_inv", C.c_void_p), ("obs", C.c_void_p),
        ("prev_coverage", C.c_void_p), ("num_steps", C.c_void_p), ("num_sim_steps", C.c_void_p),
        ("reward", C.c_void_p), ("done", C.c_void_p),
        ("iters_up_env", C.c_void_p), ("env_order", C.c_void_p),
        ("cost", C.c_void_p), ("sched_scratch", C.c_void_p), ("sched_scratch_bytes", C.c_int64),
    ]


class Physics(C.Structure):
    """ClothB200Physics: one environment's material (the `_phys` entry points take a device array of these)."""
    _fields_ = [("density", C.c_double), ("ks", C.c_double), ("damping", C.c_double), ("plane_friction", C.c_double),
                ("tear_thresh", C.c_double), ("gravity", C.c_double), ("reserved", C.c_double * 2)]


# the fields of a ClothB200Physics row, in order (a [n_env, 8] float64 tensor holds them and two zero columns)
PHYSICS_FIELDS = ("density", "ks", "damping", "plane_friction", "tear_thresh", "gravity")


class Scene(C.Structure):
    """ClothB200Scene: the Blender scene of gym_cloth/blender/get_image_rep_279.py."""
    _f3 = C.c_float * 3
    _fields_ = [
        ("height", C.c_int32), ("width", C.c_int32), ("samples", C.c_int32), ("reserved", C.c_int32),
        ("lens_mm", C.c_float), ("sensor_mm", C.c_float),
        ("cam_pos", _f3), ("cam_deg", _f3), ("lamp_pos", _f3),
        ("lamp_energy", C.c_float), ("diffuse_intensity", C.c_float), ("horizon", C.c_float),
        ("bed_z", C.c_float), ("bed_x0", C.c_float), ("bed_x1", C.c_float), ("bed_y0", C.c_float), ("bed_y1", C.c_float),
        ("floor_z", C.c_float), ("floor_x0", C.c_float), ("floor_x1", C.c_float), ("floor_y0", C.c_float), ("floor_y1", C.c_float),
        ("front", _f3), ("back", _f3), ("bed", _f3),
    ]


class SceneEnv(C.Structure):
    """ClothB200SceneEnv: optional per-environment scene values (device pointers)."""
    _fields_ = [("cam_pos_offset", C.c_void_p), ("cam_deg", C.c_void_p), ("front", C.c_void_p), ("back", C.c_void_p),
                ("bed", C.c_void_p), ("swap_sides", C.c_void_p)]


# name -> (restype, argtypes); `None` suffix-expanded for _f32/_f64
_vp, _i, _d, _i64 = C.c_void_p, C.c_int, C.c_double, C.c_int64
_PP, _SP = C.POINTER(Params), C.POINTER(Step)
_ScP, _SeP = C.POINTER(Scene), C.POINTER(SceneEnv)
_PROTOS = {
    "clothb200_version": (_i, []),
    "clothb200_error_string": (C.c_char_p, [_i]),
    "clothb200_last_cuda_error": (C.c_char_p, []),
    "clothb200_sizeof_params": (C.c_size_t, []),
    "clothb200_sizeof_plan": (C.c_size_t, []),
    "clothb200_sizeof_step": (C.c_size_t, []),
    "clothb200_sizeof_physics": (C.c_size_t, []),
    "clothb200_device_info": (_i, [_i] + [C.POINTER(C.c_int)] * 4),
    "clothb200_occupancy": (_i, [_PP, _i] + [C.POINTER(C.c_int)] * 3),
    "clothb200_step_kernel_info": (_i, [_PP, _i, _i, _i, _i] + [C.POINTER(C.c_int)] * 4),
    "clothb200_params_default": (_i, [_PP]),
    "clothb200_params_validate": (_i, [_PP]),
    "clothb200_decode_actions_host": (_i, [_PP, _i, _vp, _vp]),
    "clothb200_bench_smem_bandwidth": (_i, [_i, C.POINTER(_d), _vp]),
    "clothb200_bench_fp32_flops": (_i, [_i, C.POINTER(_d), _vp]),
    "clothb200_launch_count": (_i64, []),
    "clothb200_debug_set_profile": (_i, [_vp]),
    "clothb200_sched_scratch_bytes": (C.c_size_t, [_i]),
    "clothb200_debug_set_slicing": (_i, [_i, _i]),
    "clothb200_sizeof_scene": (C.c_size_t, []),
    "clothb200_scene_default": (_i, [_ScP]),
    "clothb200_post_depth": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "clothb200_post_rgb": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp]),
}
_TYPED = {
    "clothb200_init_grid": (_i, [_PP, _i, _vp, _i, _vp, _vp, _vp]),
    "clothb200_broadcast_state": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp]),
    "clothb200_decode_actions": (_i, [_PP, _i, _vp, _vp, _vp]),
    "clothb200_step_plans": (_i, [_PP, _i, _i, _vp, _SP, _i, _vp]),
    "clothb200_step_actions": (_i, [_PP, _i, _i, _vp, _vp, _SP, _i, _vp]),
    "clothb200_update_n": (_i, [_PP, _i, _i, _i, _SP, _vp]),
    "clothb200_grab_top": (_i, [_PP, _i, _vp, _d, _SP, _vp]),
    "clothb200_gripper_adjust": (_i, [_i, _i, _d, _d, _d, _vp, _vp, _vp]),
    "clothb200_gripper_release": (_i, [_i, _i, _vp, _vp, _vp]),
    "clothb200_measure": (_i, [_PP, _i, _SP, _vp]),
    "clothb200_step_host": (_i, [_PP, _i, _i, _vp, _SP, _i] + [_vp] * 8),
    "clothb200_step_plans_phys": (_i, [_PP, _i, _i, _vp, _SP, _i, _vp, _vp]),
    "clothb200_step_actions_phys": (_i, [_PP, _i, _i, _vp, _vp, _SP, _i, _vp, _vp]),
    "clothb200_update_n_phys": (_i, [_PP, _i, _i, _i, _SP, _vp, _vp]),
    "clothb200_step_host_phys": (_i, [_PP, _i, _i, _vp, _SP, _i] + [_vp] * 9),
    "clothb200_render_rgb": (_i, [_PP, _ScP, _SeP, _i, _vp, _vp, _vp]),
    "clothb200_render_depth": (_i, [_PP, _ScP, _SeP, _i, _vp, _vp, _vp, _vp, _vp]),
}


def exported_symbols():
    """Every symbol include/clothb200.h declares."""
    names = list(_PROTOS)
    for base in _TYPED:
        names += [base + "_f32", base + "_f64"]
    return names


_lib = None
_variants = {}
LIB_IEEE_PATH = os.path.join(HERE, "libclothb200_f32ieee.so")


def lib(variant=None):
    """The shared library.  variant='f32ieee': the study build of the f32 kernels (reference expressions, IEEE div/sqrt,
    no flush-to-zero; `python -m gym_cloth_b200.build --ieee`) - loaded side by side, used by scripts/f32_drift.py and
    the drift test only."""
    global _lib
    if variant is None and _lib is not None:
        return _lib
    if variant is not None and variant in _variants:
        return _variants[variant]
    path = LIB_PATH if variant is None else {"f32ieee": LIB_IEEE_PATH}[variant]
    if not os.path.exists(path):
        raise ClothB200Error(
            "%s is not built. Run `python -m gym_cloth_b200.build%s`; there is no CPU fallback." % (path, "" if variant is None else " --ieee"))
    L = C.CDLL(path)
    for name, (res, args) in _PROTOS.items():
        f = getattr(L, name); f.restype = res; f.argtypes = args
    for base, (res, args) in _TYPED.items():
        for sfx in ("_f32", "_f64"):
            f = getattr(L, base + sfx); f.restype = res; f.argtypes = args
    assert L.clothb200_sizeof_params() == C.sizeof(Params), "Params layout mismatch"
    assert L.clothb200_sizeof_plan() == C.sizeof(Plan), "Plan layout mismatch"
    assert L.clothb200_sizeof_step() == C.sizeof(Step), "Step layout mismatch"
    assert L.clothb200_sizeof_scene() == C.sizeof(Scene), "Scene layout mismatch"
    assert L.clothb200_sizeof_physics() == C.sizeof(Physics), "Physics layout mismatch"
    if variant is None:
        _lib = L
    else:
        _variants[variant] = L
    return L


def check(rc, what=""):
    if rc != OK:
        L = lib()
        msg = L.clothb200_error_string(rc).decode()
        if rc == -3:
            msg += ": " + L.clothb200_last_cuda_error().decode()
        raise ClothB200Error("%s failed: %s" % (what or "clothb200 call", msg), rc)


def default_params():
    P = Params()
    check(lib().clothb200_params_default(C.byref(P)), "params_default")
    return P


def default_scene():
    S = Scene()
    check(lib().clothb200_scene_default(C.byref(S)), "scene_default")
    return S


def params_from_cfg(cfg):
    """ClothB200Params from the dict the reference loads from cfg/*.yaml (cloth_env.py:87-117).

    Raises the exception types the reference raises for bad configs (cloth.pyx:85, 91, 132)."""
    P = default_params()
    cl, env = cfg["cloth"], cfg["env"]
    pin_cond = cl.get("pin_cond", "default")
    if pin_cond not in ("y=0", "x=0,y=0", "y=0,x=0", "default"):
        raise ValueError(pin_cond)                       # cloth.pyx:85 (parsed, never applied: App. B-2)
    if cfg["init"]["type"] not in INIT_TIER:
        raise ValueError(cfg["init"]["type"])            # cloth.pyx:132
    assert cl["num_height_points"] == cl["num_width_points"]   # cloth.pyx:91
    P.num_width_points = cl["num_width_points"]; P.num_height_points = cl["num_height_points"]
    P.width = cl["width"]; P.height = cl["height"]
    P.density = cl["density"]; P.ks = cl["ks"]; P.damping = cl["damping"]
    P.thickness = cl["thickness"]; P.plane_friction = cl["plane_friction"]; P.tear_thresh = cl["tear_thresh"]
    P.frames_per_sec = cfg["frames_per_sec"]; P.simulation_steps = cfg["simulation_steps"]
    P.iters_up = env["iters_up"]; P.iters_up_rest = env["iters_up_rest"]
    P.iters_grip_rest = env["iters_grip_rest"]; P.iters_rest = env["iters_rest"]
    P.iters_pull_max = env["iters_pull_max"]; P.max_actions = env["max_actions"]
    P.reduce_factor = env["reduce_factor"]; P.grip_radius = env["grip_radius"]
    P.gripper_height = cl["height"]                      # Gripper(cloth, grip_radius, cfg.cloth.height, ...) cloth_env.py:752
    P.clip_act_space = int(bool(env["clip_act_space"])); P.delta_actions = int(bool(env["delta_actions"]))
    P.force_grab = int(bool(env.get("force_grab", False)))
    rt = env.get("reward_type", "coverage-delta")
    assert "coverage" in rt                              # cloth_env.py:130
    if rt not in REWARD_TYPE:
        raise ValueError(rt)                             # cloth_env.py:679 (the height/variance types fail the assert above)
    P.reward_type = REWARD_TYPE[rt]
    check(lib().clothb200_params_validate(C.byref(P)), "params_validate")
    return P


def physics_of(P):
    """The material of ClothB200Params P as a dict of the ClothB200Physics fields."""
    return {k: float(getattr(P, k)) for k in PHYSICS_FIELDS}


def copy_params(P):
    Q = Params()
    C.memmove(C.byref(Q), C.byref(P), C.sizeof(Params))
    return Q
