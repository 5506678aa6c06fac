"""BatchedCloth: n independent cloths resident in HBM, stepped by the sm_100a kernels.

PyTorch is used for what it is good at here - owning device memory and streams.  All arithmetic
happens inside libclothb200.so (gym_cloth_b200/csrc).  State layout (include/clothb200.h):
    pos [n_env, N, 4] = (x, y, z, pinned)          prev[n_env, N, 4] = (px, py, pz, grab multiplicity)
"""
import ctypes as C

import numpy as np
import torch

from . import lib as _l


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class BatchedCloth(object):
    """The batched counterpart of the reference's Cloth + Gripper pair (gym_cloth/physics/cloth.pyx,
    gripper.pyx) for `n_env` independent environments on one GPU."""

    def __init__(self, params, n_env, dtype=torch.float32, device=None, init_type="tier1", noise=None,
                 init_side=True, exact_rest=None, mode=_l.MODE_REFERENCE_ORDER, variant=None):
        if not torch.cuda.is_available():
            raise _l.ClothB200Error("BatchedCloth needs a CUDA device (no CPU fallback)")
        self.L = _l.lib(variant)
        self.P = params
        self.n_env = int(n_env)
        self.dtype = dtype
        assert dtype in (torch.float32, torch.float64)
        self.sfx = "_f32" if dtype == torch.float32 else "_f64"
        self.device = torch.device(device if device is not None else "cuda")
        self.mode = mode
        self.W = params.num_width_points
        self.N = self.W * params.num_height_points
        self.nwords = (self.N + 31) // 32
        n, N, dev = self.n_env, self.N, self.device
        z = lambda *s, dt=torch.int32: torch.zeros(*s, dtype=dt, device=dev)
        self.pos = z(n, N, 4, dt=dtype); self.prev = z(n, N, 4, dt=dtype)
        self.flags = z(n); self.sim_steps = z(n); self.n_grabbed = z(n)
        self.grab_mask = z(n, self.nwords)
        self.coverage = z(n, dt=torch.float64); self.variance_inv = z(n, dt=torch.float64)
        self.obs = z(n, 3 * N, dt=dtype)
        self.prev_coverage = z(n, dt=torch.float64)
        self.num_steps = z(n); self.num_sim_steps = z(n)
        self.reward = z(n, dt=torch.float64); self.done = z(n)
        self.plans = torch.zeros(n, C.sizeof(_l.Plan), dtype=torch.uint8, device=dev)
        # measured cycles/substep per env (diagnostics) + scratch for the on-device launch order and the time-sliced queue
        self.cost = torch.zeros(n, dtype=torch.float32, device=dev)
        self.sched_scratch = torch.zeros(int(self.L.clothb200_sched_scratch_bytes(max(n, 1))), dtype=torch.uint8, device=dev)
        self.schedule = True
        self.time_slice = True         # False: one CTA runs a whole action (ClothB200Step.sched_scratch_bytes = 0)
        self.iters_up_env = None
        self.env_order = None
        self.rest = None
        self.rest_env_stride = 0
        # per-environment material: None = every cloth runs params' material; else [n_env, 8] float64 on the device,
        # one ClothB200Physics row per environment (lib.PHYSICS_FIELDS, then two zeros)
        self.physics = None
        # the parity build always uses the exact per-spring rest lengths; f32 tier-1/3 can use constants
        if exact_rest is None:
            exact_rest = (dtype == torch.float64) or init_type == "tier2"
        self.exact_rest = exact_rest
        self.reset_grid(init_type, noise, init_side)

    # ------------------------------------------------------------------ helpers
    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _np_dtype(self):
        return np.float32 if self.dtype == torch.float32 else np.float64

    def _f(self, base):
        """The typed entry point, called with this batch's device current (launches, attribute caches and scratch
        buffers of the library all belong to the current device)."""
        fn = getattr(self.L, base + self.sfx)
        dev = self.device

        def call(*args):
            with torch.cuda.device(dev):
                return fn(*args)
        return call

    def io(self, measure=True, bookkeeping=True, obs=True, grab_mask=True):
        s = _l.Step()
        s.pos = self.pos.data_ptr(); s.prev = self.prev.data_ptr()
        s.rest = self.rest.data_ptr() if self.rest is not None else None
        s.rest_env_stride = self.rest_env_stride
        s.flags = self.flags.data_ptr(); s.sim_steps = self.sim_steps.data_ptr()
        s.n_grabbed = self.n_grabbed.data_ptr()
        s.grab_mask = self.grab_mask.data_ptr() if grab_mask else None
        if measure:
            s.coverage = self.coverage.data_ptr(); s.variance_inv = self.variance_inv.data_ptr()
        s.obs = self.obs.data_ptr() if obs else None
        if bookkeeping:
            s.prev_coverage = self.prev_coverage.data_ptr(); s.num_steps = self.num_steps.data_ptr()
            s.num_sim_steps = self.num_sim_steps.data_ptr(); s.reward = self.reward.data_ptr()
            s.done = self.done.data_ptr()
        s.iters_up_env = self.iters_up_env.data_ptr() if self.iters_up_env is not None else None
        s.env_order = self.env_order.data_ptr() if self.env_order is not None else None
        s.cost = self.cost.data_ptr()
        s.sched_scratch = self.sched_scratch.data_ptr() if (self.schedule and self.env_order is None) else None
        s.sched_scratch_bytes = self.sched_scratch.numel() if self.time_slice else 0
        return s

    # ------------------------------------------------------------------ construction (Cloth.__init__)
    def reset_grid(self, init_type="tier1", noise=None, init_side=True, envs=None):
        """Cloth.__init__ grid (cloth.pyx:92-130) for all (or the given) environments.
        noise: [N] or [n_sel, N] doubles as drawn by the reference (tier2)."""
        npdt = self._np_dtype()
        N = self.N
        tier = _l.INIT_TIER[init_type] if isinstance(init_type, str) else int(init_type)
        sel = None if envs is None else torch.as_tensor(envs, device=self.device, dtype=torch.long)
        n_sel = self.n_env if sel is None else int(sel.numel())
        per_env = noise is not None and np.ndim(noise) == 2
        count = n_sel if per_env else 1
        pos4 = np.zeros((count, N, 4), npdt); prev4 = np.zeros((count, N, 4), npdt); rest6 = np.zeros((count, 6 * N), npdt)
        sides = np.broadcast_to(np.asarray(init_side, dtype=bool), (count,))
        for i in range(count):
            nz = None
            if noise is not None:
                nz = np.ascontiguousarray(noise[i] if per_env else noise, np.float64)
            _l.check(self._f("clothb200_init_grid")(C.byref(self.P), tier, nz.ctypes.data if nz is not None else None,
                                                   int(sides[i]), pos4[i].ctypes.data, prev4[i].ctypes.data,
                                                   rest6[i].ctypes.data), "init_grid")
        tp = torch.from_numpy(pos4).to(self.device); tq = torch.from_numpy(prev4).to(self.device)
        if count == 1 and sel is None:
            _l.check(self._f("clothb200_broadcast_state")(N, self.n_env, _ptr(tp), _ptr(tq), _ptr(self.pos), _ptr(self.prev),
                                                         self.stream), "broadcast_state")
        elif sel is None:
            self.pos.copy_(tp); self.prev.copy_(tq)
        else:
            self.pos[sel] = tp.expand(n_sel, N, 4) if count == 1 else tp
            self.prev[sel] = tq.expand(n_sel, N, 4) if count == 1 else tq
        if self.exact_rest:
            tr = torch.from_numpy(rest6).to(self.device)
            if per_env:
                if self.rest is None or self.rest_env_stride == 0:
                    self.rest = torch.zeros(self.n_env, 6 * N, dtype=self.dtype, device=self.device)
                    self.rest_env_stride = 6 * N
                if sel is None:
                    self.rest.copy_(tr)
                else:
                    self.rest[sel] = tr
            elif self.rest is not None and self.rest_env_stride:
                if sel is None:
                    self.rest.copy_(tr.expand(self.n_env, 6 * N))
                else:
                    self.rest[sel] = tr.expand(n_sel, 6 * N)
            else:
                self.rest = tr.reshape(6 * N).contiguous()
                self.rest_env_stride = 0
        if sel is None:
            self.flags.zero_()
        else:
            self.flags[sel] = 0
        torch.cuda.current_stream(self.device).synchronize()   # host staging buffers go out of scope

    def set_rest(self, rest_compact, a=None, b=None, env=None):
        """Install Spring.rest_length values given in the reference's spring-list order (3502 for 25x25)."""
        W, N = self.W, self.N
        slots = spring_slots(W)
        r6 = np.zeros(6 * N, self._np_dtype())
        r6[slots] = np.asarray(rest_compact, np.float64).astype(self._np_dtype())
        t = torch.from_numpy(r6).to(self.device)
        if env is None:
            self.rest = t; self.rest_env_stride = 0
        else:
            if self.rest is None or self.rest_env_stride == 0:
                base = self.rest if self.rest is not None else t
                self.rest = base.reshape(1, 6 * N).repeat(self.n_env, 1).contiguous()
                self.rest_env_stride = 6 * N
            self.rest[env] = t
        self.exact_rest = True

    def set_physics(self, envs=None, **fields):
        """Per-environment material: set the given lib.PHYSICS_FIELDS (scalars or one value per selected environment)
        for all (or the given) environments.  The first call starts every row from params' values.  Rows are not
        checked here: the kernels treat a row with a non-finite value or density <= 0 as a bad action (BADSTATE)."""
        unknown = set(fields) - set(_l.PHYSICS_FIELDS)
        if unknown:
            raise TypeError("unknown physics fields: %s" % sorted(unknown))
        if self.physics is None:
            row = [getattr(self.P, k) for k in _l.PHYSICS_FIELDS] + [0.0, 0.0]
            self.physics = torch.tensor([row], dtype=torch.float64, device=self.device).repeat(self.n_env, 1).contiguous()
        sel = slice(None) if envs is None else torch.as_tensor(np.asarray(envs, np.int64), device=self.device)
        for k, v in fields.items():
            self.physics[sel, _l.PHYSICS_FIELDS.index(k)] = torch.as_tensor(np.asarray(v, np.float64), device=self.device)

    # ------------------------------------------------------------------ state access
    def set_state(self, pos3, prev3, pinned=None, grabbed=None, env=None, tear=False):
        """Load one state (N x 3 arrays, pinned [N] bool, grabbed = index list with multiplicity)
        into environment `env` (or all environments)."""
        N = self.N
        p4 = np.zeros((N, 4), np.float64); q4 = np.zeros((N, 4), np.float64)
        p4[:, :3] = pos3; q4[:, :3] = prev3
        if pinned is not None:
            p4[:, 3] = np.asarray(pinned, np.float64)
        if grabbed is not None and len(grabbed):
            np.add.at(q4[:, 3], np.asarray(grabbed, np.int64), 1.0)
        tp = torch.from_numpy(p4).to(self.device, self.dtype); tq = torch.from_numpy(q4).to(self.device, self.dtype)
        if env is None:
            self.pos.copy_(tp.expand(self.n_env, N, 4)); self.prev.copy_(tq.expand(self.n_env, N, 4))
            self.flags.fill_(_l.FLAG_TEAR if tear else 0)
        else:
            self.pos[env] = tp; self.prev[env] = tq
            self.flags[env] = _l.FLAG_TEAR if tear else 0

    def get_state(self, env=0):
        p = self.pos[env].double().cpu().numpy(); q = self.prev[env].double().cpu().numpy()
        return p[:, :3].copy(), q[:, :3].copy(), (p[:, 3] != 0), q[:, 3].astype(np.int64)

    def grabbed_set(self, env=0):
        """Indices with a set bit in the grab mask written by the last grab_top/step."""
        words = self.grab_mask[env].cpu().numpy().view(np.uint32)
        bits = np.unpackbits(words.view(np.uint8), bitorder="little")[: self.N]
        return np.nonzero(bits)[0]

    # ------------------------------------------------------------------ the hot path
    def update(self, n_updates=1, measure=False):
        """n x Cloth.update() (cloth.pyx:169-214)."""
        io = self.io(measure=measure, bookkeeping=False, obs=False, grab_mask=False)
        if self.physics is not None:
            _l.check(self._f("clothb200_update_n_phys")(C.byref(self.P), self.mode, self.n_env, int(n_updates), C.byref(io),
                                                       _ptr(self.physics), self.stream), "update_n_phys")
            return
        _l.check(self._f("clothb200_update_n")(C.byref(self.P), self.mode, self.n_env, int(n_updates), C.byref(io),
                                              self.stream), "update_n")

    def decode_host(self, actions):
        """cloth_env.py:401-470 on the host with CPython's exact arithmetic; returns a ctypes Plan array."""
        a = np.ascontiguousarray(actions, np.float64).reshape(-1, 4)
        plans = (_l.Plan * len(a))()
        _l.check(self.L.clothb200_decode_actions_host(C.byref(self.P), len(a), a.ctypes.data, C.addressof(plans)), "decode_host")
        return plans

    def step_plans(self, plans, initialize=False, measure=True, obs=True):
        """plans: ctypes (Plan * n_env) array (host) or a uint8 device tensor of packed plans."""
        if not isinstance(plans, torch.Tensor):
            host = torch.frombuffer(bytearray(bytes(plans)), dtype=torch.uint8).reshape(self.n_env, C.sizeof(_l.Plan))
            self.plans.copy_(host)
            plans = self.plans
        io = self.io(measure=measure, bookkeeping=not initialize, obs=obs)
        if self.physics is not None:
            _l.check(self._f("clothb200_step_plans_phys")(C.byref(self.P), self.mode, self.n_env, _ptr(plans), C.byref(io),
                                                         int(initialize), _ptr(self.physics), self.stream), "step_plans_phys")
            return
        _l.check(self._f("clothb200_step_plans")(C.byref(self.P), self.mode, self.n_env, _ptr(plans), C.byref(io),
                                                int(initialize), self.stream), "step_plans")

    def step_actions(self, actions, initialize=False, measure=True, obs=True):
        """actions: device tensor [n_env, 4] of this cloth's dtype, env.step format.  Decode on device."""
        assert actions.is_cuda and actions.dtype == self.dtype and actions.is_contiguous()
        io = self.io(measure=measure, bookkeeping=not initialize, obs=obs)
        if self.physics is not None:
            _l.check(self._f("clothb200_step_actions_phys")(C.byref(self.P), self.mode, self.n_env, _ptr(actions),
                                                           _ptr(self.plans), C.byref(io), int(initialize), _ptr(self.physics),
                                                           self.stream), "step_actions_phys")
            return
        _l.check(self._f("clothb200_step_actions")(C.byref(self.P), self.mode, self.n_env, _ptr(actions), _ptr(self.plans),
                                                  C.byref(io), int(initialize), self.stream), "step_actions")

    def step_host(self, actions, out, initialize=False):
        """Host-buffer entry point: actions np.float64 [n_env,4]; `out` dict of (ideally pinned) host
        arrays among obs/reward/done/coverage/variance_inv/flags/sim_steps.  Synchronous."""
        a = np.ascontiguousarray(actions, np.float64)
        io = self.io(measure=True, bookkeeping=not initialize, obs=("obs" in out))
        g = lambda k: C.c_void_p(out[k].ctypes.data if isinstance(out[k], np.ndarray) else out[k].data_ptr()) if k in out else None
        if self.physics is not None:
            _l.check(self._f("clothb200_step_host_phys")(C.byref(self.P), self.mode, self.n_env, a.ctypes.data, C.byref(io),
                                                        int(initialize), g("obs"), g("reward"), g("done"), g("coverage"),
                                                        g("variance_inv"), g("flags"), g("sim_steps"), _ptr(self.physics),
                                                        self.stream), "step_host_phys")
            return
        _l.check(self._f("clothb200_step_host")(C.byref(self.P), self.mode, self.n_env, a.ctypes.data, C.byref(io), int(initialize),
                                               g("obs"), g("reward"), g("done"), g("coverage"), g("variance_inv"), g("flags"),
                                               g("sim_steps"), self.stream), "step_host")

    # ------------------------------------------------------------------ pieces
    def grab_top(self, xy, grip_radius=None):
        xy_t = torch.as_tensor(np.broadcast_to(np.asarray(xy, np.float64), (self.n_env, 2)).copy(), device=self.device)
        io = self.io(measure=False, bookkeeping=False, obs=False)
        r = self.P.grip_radius if grip_radius is None else float(grip_radius)
        _l.check(self._f("clothb200_grab_top")(C.byref(self.P), self.n_env, _ptr(xy_t), r, C.byref(io), self.stream), "grab_top")
        torch.cuda.current_stream(self.device).synchronize()

    def adjust(self, x, y, z):
        _l.check(self._f("clothb200_gripper_adjust")(self.N, self.n_env, float(x), float(y), float(z), _ptr(self.pos),
                                                    _ptr(self.prev), self.stream), "gripper_adjust")

    def release(self):
        _l.check(self._f("clothb200_gripper_release")(self.N, self.n_env, _ptr(self.pos), _ptr(self.prev), self.stream),
                 "gripper_release")

    def measure(self):
        io = self.io(measure=True, bookkeeping=False, obs=True)
        _l.check(self._f("clothb200_measure")(C.byref(self.P), self.n_env, C.byref(io), self.stream), "measure")


_SLOT_CACHE = {}


def spring_slots(W):
    """Slot index q*6+k of every spring in the reference's creation order (cloth.pyx:135-146)."""
    if W in _SLOT_CACHE:
        return _SLOT_CACHE[W]
    out = []
    for r in range(W):
        for c in range(W):
            q = r * W + c
            ok = (r > 0, c > 0, r > 0 and c > 0, r > 0 and c + 1 < W, r > 1, c > 1)
            out += [q * 6 + k for k in range(6) if ok[k]]
    _SLOT_CACHE[W] = np.array(out, np.int64)
    return _SLOT_CACHE[W]
