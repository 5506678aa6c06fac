"""Host-side mirror of gym_cloth/envs/cloth_env.py for the B200 path.

`BatchedClothEnv`  n independent ClothEnv instances on one GPU (vector-env API).
`ClothEnv`         single-env facade with the reference's constructor, method and attribute names
                   (cloth_env.py:55-1228), so that scripts such as examples/analytic.py keep working.

All arithmetic of the hot path (Cloth.update, Gripper, the substep loop, coverage/reward/terminal)
runs in libclothb200.so; this file holds only what the reference also does in Python: config handling,
random draws for resets and the gym-style bookkeeping.  Random numbers are drawn from
np.random.RandomState streams in exactly the order the reference draws them, environment i seeded like
the reference's `env.seed(seed + i)` (gym 0.12.1 seeding, gym_cloth_b200/seeding.py), so environment i replays the
reference ClothEnv seeded with seed + i (bit-exactly in f64).  The reference also draws 3 + 224*224*3 values of
per-episode domain randomisation from the same stream at the end of every reset (cloth_env.py:786-789), whatever the
observation type: the single-env `ClothEnv` facade replays them (every episode matches), `BatchedClothEnv` does so
only with dom_rand_draws=True (otherwise its FIRST episode per environment matches and later ones use their own,
equally distributed, draws - 150 531 draws per reset and environment are not free at 65 536 environments).
"""
import copy
import pickle

import contextlib

import numpy as np
import torch
import yaml

from .. import lib as _l
from .. import seeding as _seeding
from ..batched import BatchedCloth

_REWARD_THRESHOLDS = {"coverage": 0.92, "coverage-delta": 0.92}   # cloth_env.py:42-50 (coverage types only)


def load_cfg(cfg):
    if isinstance(cfg, dict):
        return copy.deepcopy(cfg)
    with open(cfg, "r") as fh:
        return yaml.safe_load(fh)


class _Box(object):
    """The two attributes of gym.spaces.Box that ClothEnv users touch (cloth_env.py:148-181)."""

    def __init__(self, low, high, dtype=np.float32):
        self.low = np.asarray(low, dtype=dtype); self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape; self.dtype = np.dtype(dtype)
        self.np_random = np.random.RandomState()

    def seed(self, seed=None):
        self.np_random = np.random.RandomState(seed); return [seed]

    def sample(self):
        return self.np_random.uniform(self.low, self.high, size=self.shape).astype(self.dtype)


def _randval_minabs(rs, low, high, minabs=None):   # cloth_env.py:825-833
    val = rs.uniform(low=low, high=high)
    if minabs is not None:
        while np.abs(val) < minabs:
            val = rs.uniform(low=low, high=high)
    return val


def _prevent_oob(val, dval, lower=0.0, upper=1.0):   # cloth_env.py:835-841
    if val + dval < lower:
        dval = lower - val
    elif val + dval > upper:
        dval = upper - val
    return dval


class BatchedClothEnv(object):
    """n_env ClothEnv instances stepped by one kernel launch per env.step.

    actions: [n_env, 4] in env.step's format (cfg clip_act_space/delta_actions as in cfg/t*_rgbd.yaml).
    Global environment ids are env_offset + i (multi-GPU shards pass their offset) and only seed the RNG
    streams, so results do not depend on how the batch is sharded.
    """

    def __init__(self, cfg, n_env, dtype="f32", device=None, seed=None, env_offset=0, dom_rand_draws=False,
                 mode=_l.MODE_REFERENCE_ORDER, physics=None):
        self.cfg = load_cfg(cfg)
        cfg = self.cfg
        self.P = _l.params_from_cfg(cfg)
        env = cfg["env"]
        self.obs_type = env["obs_type"]
        if self.obs_type not in ("1d", "blender"):
            raise ValueError(self.obs_type)              # cloth_env.py:155-156
        # image observations (cloth_env.py:107-117): the flags are the strings 'True' / 'False' in the cfg
        self.use_depth = str(env.get("use_depth", "False")) == "True"
        self.use_rgbd = str(env.get("use_rgbd", "False")) == "True"
        self.add_dom_rand = str(env.get("use_dom_rand", "False")).lower() == "true"
        self.reward_type = env["reward_type"]
        assert "coverage" in self.reward_type             # cloth_env.py:130
        if self.reward_type not in _REWARD_THRESHOLDS:
            raise ValueError(self.reward_type)            # cloth_env.py:679
        if not (env["clip_act_space"] and env["delta_actions"]):
            raise NotImplementedError("reset actions need delta_actions (cloth_env.py:861-862)")
        self.init_type = cfg["init"]["type"]
        self.n_env = int(n_env)
        self.env_offset = int(env_offset)
        self.torch_dtype = torch.float32 if dtype in ("f32", torch.float32) else torch.float64
        self.max_actions = env["max_actions"]
        self.grip_radius = env["grip_radius"]
        self.dom_rand_draws = dom_rand_draws
        self.time_resets = False          # True: reset() leaves the GPU's own busy time of the reset in reset_device_ms
        self.N = self.P.num_width_points * self.P.num_height_points
        self.action_space = _Box([-1., -1., -1., -1.], [1., 1., 1., 1.])
        lim = 100
        self.observation_space = _Box(-lim * np.ones(3 * self.N), lim * np.ones(3 * self.N))
        self.cloth = BatchedCloth(self.P, self.n_env, dtype=self.torch_dtype, device=device,
                                  init_type="tier1" if self.init_type == "tier3" else self.init_type,
                                  noise=np.zeros(self.N) if self.init_type == "tier2" else None, mode=mode)
        self.device = self.cloth.device
        self.renderer = None
        if self.obs_type == "blender":
            from ..render import ClothRenderer
            self.renderer = ClothRenderer(self.P, self.n_env, device=self.device)
            hd, wd = self.renderer.H, self.renderer.W
            self.observation_space = _Box(np.zeros((hd, wd, 3)), np.ones((hd, wd, 3)), dtype=np.uint8)   # cloth_env.py:149-154
            self._dr = {"gval_depth": np.full(self.n_env, 50.0, np.float32), "gval_rgb": np.ones(self.n_env),
                        "c": np.ones((self.n_env, 3), np.float32), "n1": np.zeros((self.n_env, 3), np.float32),
                        "camera_pos": np.zeros((self.n_env, 3), np.float32), "camera_deg": np.zeros((self.n_env, 3), np.float32)}
            self._noise = None
        self.init_side = np.ones(self.n_env, bool)
        self.start_coverage = torch.zeros(self.n_env, dtype=torch.float64, device=self.device)
        self.start_variance_inv = torch.zeros(self.n_env, dtype=torch.float64, device=self.device)
        self._pinned = None
        if physics is not None:
            self.set_physics(**physics)
        self.seed(cfg.get("seed", 0) if seed is None else seed)

    # ------------------------------------------------------------------ per-environment material
    def get_physics(self):
        """The material of every environment: dict of float64 arrays [n_env] (lib.PHYSICS_FIELDS)."""
        if self.cloth.physics is None:
            return {k: np.full(self.n_env, float(getattr(self.P, k))) for k in _l.PHYSICS_FIELDS}
        t = self.cloth.physics.cpu().numpy()
        return {k: t[:, i].copy() for i, k in enumerate(_l.PHYSICS_FIELDS)}

    def set_physics(self, envs=None, density=None, ks=None, damping=None, plane_friction=None, tear_thresh=None, gravity=None):
        """Give the selected environments (all by default) their own material: each value a scalar or one value per
        selected environment; a field left None keeps its current value (initially the cfg's).  The values persist
        across reset(), whose pulls and settle loops run under each environment's own material.  Raises ValueError for
        a wrong length, a non-finite value or density <= 0."""
        sel = self._sel(envs)
        if len(sel) and (sel.min() < 0 or sel.max() >= self.n_env):
            raise ValueError("environment index out of range")
        given = {k: v for k, v in (("density", density), ("ks", ks), ("damping", damping), ("plane_friction", plane_friction),
                                   ("tear_thresh", tear_thresh), ("gravity", gravity)) if v is not None}
        new = {}
        for k, v in given.items():
            a = np.asarray(v, np.float64)
            if a.ndim == 0:
                a = np.full(len(sel), float(a))
            if a.shape != (len(sel),):
                raise ValueError("%s: expected a scalar or %d values, got shape %s" % (k, len(sel), a.shape))
            if not np.all(np.isfinite(a)):
                raise ValueError("%s: values must be finite" % k)
            if k == "density" and not np.all(a > 0):
                raise ValueError("density must be > 0")
            new[k] = a
        if new:
            self.cloth.set_physics(envs=sel, **new)

    # ------------------------------------------------------------------ seeding
    def seed(self, seed=None):
        """Environment i draws from the generator `ClothEnv.seed(seed + env_offset + i)` creates in the reference
        (cloth_env.py:332-341): gym 0.12.1's seeding.np_random, i.e. MT19937 keyed by the SHA-512 hash of the seed."""
        if seed is None:
            seed = _seeding.create_seed() % (2 ** 31)
        self._seed = int(seed)
        self.rngs = [_seeding.np_random(self._seed + self.env_offset + i)[0] for i in range(self.n_env)]
        return [seed]

    # ------------------------------------------------------------------ helpers
    def _sel(self, envs):
        if envs is None:
            return np.arange(self.n_env)
        return np.asarray(envs, np.int64).reshape(-1)

    def _points_xy(self, envs, pidx):
        """(x, y) of point pidx[j] of environment envs[j] as Python-exact doubles."""
        e = torch.as_tensor(envs, device=self.device); p = torch.as_tensor(pidx, device=self.device)
        return self.cloth.pos[e, p, :2].double().cpu().numpy()

    @contextlib.contextmanager
    def _timed(self):
        """CUDA events around one device call of a reset (reset_device_ms: how long the GPU itself worked)."""
        ev = getattr(self, "_reset_events", None)
        if ev is None:
            yield
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        yield
        b.record()
        ev.append((a, b))

    def _step_subset(self, envs, actions, initialize, iters_up=None):
        """step(action, initialize) for a subset of environments (host decode = CPython arithmetic)."""
        c = self.cloth
        full = np.zeros((self.n_env, 4))
        full[envs] = actions
        plans = c.decode_host(full)
        order = torch.as_tensor(envs, dtype=torch.int32, device=self.device)
        old_order, old_n, old_iu = c.env_order, c.n_env, c.iters_up_env
        if iters_up is not None:
            iu = np.full(self.n_env, float(self.P.iters_up)); iu[envs] = iters_up
            c.iters_up_env = torch.from_numpy(iu).to(self.device)
        host = torch.frombuffer(bytearray(bytes(plans)), dtype=torch.uint8).reshape(self.n_env, -1)
        c.plans.copy_(host)
        c.env_order, c.n_env = order, len(envs)
        try:
            with self._timed():
                c.step_plans(c.plans, initialize=initialize)
        finally:
            c.env_order, c.n_env, c.iters_up_env = old_order, old_n, old_iu

    def _update_subset(self, envs, n_updates):
        c = self.cloth
        order = torch.as_tensor(envs, dtype=torch.int32, device=self.device)
        old_order, old_n = c.env_order, c.n_env
        c.env_order, c.n_env = order, len(envs)
        try:
            with self._timed():
                c.update(n_updates)
        finally:
            c.env_order, c.n_env = old_order, old_n

    def _measure_subset(self, envs):
        c = self.cloth
        order = torch.as_tensor(envs, dtype=torch.int32, device=self.device)
        old_order, old_n = c.env_order, c.n_env
        c.env_order, c.n_env = order, len(envs)
        try:
            c.measure()
        finally:
            c.env_order, c.n_env = old_order, old_n
        torch.cuda.current_stream(self.device).synchronize()

    # ------------------------------------------------------------------ reset (cloth_env.py:717-987)
    def reset(self, envs=None):
        """Start a new episode in the given environments (all by default).  Returns obs [n_env, 3N]."""
        envs = self._sel(envs)
        c = self.cloth
        n = len(envs)
        if n == 0:
            return c.obs
        self._reset_events = [] if self.time_resets else None
        # Cloth.__init__ (cloth.pyx:75, 94-130): init_side is always drawn, tier2 draws the x-noise
        sides = np.array([self.rngs[e].rand() > 0.5 for e in envs])
        self.init_side[envs] = sides
        if self.init_type == "tier2":
            noise = np.stack([self.rngs[e].rand(self.N) * 0.01 - 0.005 for e in envs])
            c.reset_grid("tier2", noise=noise, init_side=sides, envs=envs)
        else:
            c.reset_grid("tier1", envs=envs)
        idx_t = torch.as_tensor(envs, device=self.device)
        c.num_steps[idx_t] = 0; c.num_sim_steps[idx_t] = 0
        if getattr(self, "orig_pos", None) is None:
            self.orig_pos = torch.zeros(self.n_env, self.N, 3, dtype=torch.float64, device=self.device)
        self.orig_pos[idx_t] = c.pos[idx_t, :, :3].double()       # Point.orig_x/y/z (point.pyx: set once at construction)
        self.init_actions = {int(e): [] for e in envs}
        self._reset_actions(envs, sides)
        self._measure_subset(envs)
        self.start_coverage[idx_t] = c.coverage[idx_t]
        self.start_variance_inv[idx_t] = c.variance_inv[idx_t]
        c.prev_coverage[idx_t] = c.coverage[idx_t]
        if self.dom_rand_draws or self.renderer is not None:
            self._draw_dom_rand(envs)
        if self._reset_events is not None:
            torch.cuda.current_stream(self.device).synchronize()
            self.reset_device_ms = sum(a.elapsed_time(b) for a, b in self._reset_events)
            self._reset_events = None
        return c.obs if self.renderer is None else self.image_obs()

    def _draw_dom_rand(self, envs):
        """Per-episode domain randomisation values, drawn in the reference's order from the reference's generators
        (cloth_env.py:786-794: the first four from the env's np_random, the rest from the global np.random).  The 1-D
        observation never uses them but the draws are replayed so that later resets see the reference's numbers."""
        keep = self.renderer is not None and self.add_dom_rand
        if keep and self._noise is None:
            self._noise = torch.zeros(self.n_env, self.renderer.H, self.renderer.W, 3, dtype=torch.float32, device=self.device)
        for e in envs:
            rs = self.rngs[e]
            gval_depth = rs.uniform(low=40, high=50); gval_rgb = rs.uniform(low=0.7, high=1.3)
            lim = rs.uniform(low=-15.0, high=15.0)
            noise = rs.uniform(low=-lim, high=lim, size=(224, 224, 3))
            # these come from the global generator in the reference, whatever the observation type (:790-794)
            c = np.random.uniform(low=0.4, high=0.6, size=(3,)); n1 = np.random.uniform(low=-0.35, high=0.35, size=(3,))
            cp = np.random.normal(0., scale=0.04, size=(3,)); cd = np.random.normal(0., scale=0.90, size=(3,))
            np.random.uniform(low=0.0, high=0.0)          # specular_max
            if keep:
                d = self._dr
                d["gval_depth"][e] = gval_depth; d["gval_rgb"][e] = gval_rgb
                d["c"][e] = c; d["n1"][e] = n1; d["camera_pos"][e] = cp; d["camera_deg"][e] = cd
                self._noise[e] = torch.from_numpy(noise.astype(np.float32)).to(self.device)
        if self.renderer is None:
            return
        r = self.renderer
        # tier2 cloths dropped from the other side show their other face (get_image_rep_279.py:236-238)
        swap = ((self.init_type == "tier2") & ~self.init_side).astype(np.int32)
        r.set_env_values(swap_sides=swap)
        if keep:
            from ..render import gamma_lut
            d = self._dr
            back = np.clip(np.array([0.070, 0.300, 0.900]) + d["n1"], 0.0, 1.0)     # get_image_rep_279.py:248-253
            front = np.clip(np.array([0.070, 0.050, 0.600]) + d["n1"], 0.0, 1.0)
            r.set_env_values(cam_pos_offset=d["camera_pos"], cam_deg=d["camera_deg"], front=front, back=back, bed=d["c"])
            self._lut = torch.from_numpy(np.stack([gamma_lut(g) for g in d["gval_rgb"]])).to(self.device)
            self._sub = torch.from_numpy(d["gval_depth"]).to(self.device)

    def image_obs(self):
        """The observation of obs_type 'blender' (cloth_env.py:201-209): uint8 [n_env, 224, 224, 3], BGR or depth,
        or [.., 4] = BGR + depth when use_rgbd."""
        r, pos = self.renderer, self.cloth.pos
        dr = self.add_dom_rand
        lut, sub, noise = (self._lut, self._sub, self._noise) if dr else (None, None, None)
        if self.use_rgbd:
            return r.rgbd(pos, lut=lut, sub=sub, noise_rgb=noise, noise_depth=noise)
        if self.use_depth:
            return r.depth(pos, sub=sub, noise=noise)
        return r.rgb(pos, lut=lut, noise=noise)

    def _clip_space(self, x, y, dx, dy):   # _convert_action_to_clip_space, cloth_env.py:1207-1215
        return ((x - 0.5) * 2, (y - 0.5) * 2, dx, dy)

    def _reset_actions(self, envs, sides):
        c = self.cloth
        n = len(envs)
        if self.init_type == "tier1":      # cloth_env.py:843-891
            lim = 0.20

            def pull(sub):
                pidx = np.array([self.rngs[e].randint(self.N) for e in sub])
                draws = [(_randval_minabs(self.rngs[e], -lim, lim, 0.08), _randval_minabs(self.rngs[e], -lim, lim, 0.08)) for e in sub]
                xy = self._points_xy(sub, pidx)
                acts = np.zeros((len(sub), 4))
                for j, e in enumerate(sub):
                    px, py = float(xy[j, 0]), float(xy[j, 1])
                    dx = _prevent_oob(px, draws[j][0]); dy = _prevent_oob(py, draws[j][1])
                    acts[j] = self._clip_space(px, py, dx, dy)
                    self.init_actions[int(e)].append(acts[j].copy())
                self._step_subset(sub, acts, initialize=True)

            pull(envs); pull(envs)
            self._measure_subset(envs)
            cov = c.coverage[torch.as_tensor(envs, device=self.device)].cpu().numpy()
            third = envs[cov >= 0.90]
            if len(third):
                pull(third)
        elif self.init_type == "tier2":    # cloth_env.py:893-949
            self._update_subset(envs, 1500)
            init_side = np.where(sides, 1, -1)
            corner = np.array([-25 if self.rngs[e].rand() < 0.5 else -1 for e in envs])
            W = self.P.num_width_points
            pidx = np.where(corner == -25, self.N - W, self.N - 1)
            dx0 = np.array([self.rngs[e].uniform(0.30, 0.50) for e in envs]) * init_side
            dy0 = np.array([self.rngs[e].uniform(0.30, 0.60) if corner[j] == -25 else self.rngs[e].uniform(-0.60, -0.30)
                            for j, e in enumerate(envs)])
            xy = self._points_xy(envs, pidx)
            acts = np.array([self._clip_space(float(xy[j, 0]), float(xy[j, 1]), dx0[j], dy0[j]) for j in range(n)])
            for j, e in enumerate(envs):
                self.init_actions[int(e)].append(acts[j].copy())
            self._step_subset(envs, acts, initialize=True)
            pidx = np.where(corner == -25, self.N - 19, self.N - 7)
            dx1 = np.array([self.rngs[e].uniform(0.30, 0.60) for e in envs]) * init_side
            dy1 = np.array([self.rngs[e].uniform(-0.30, -0.60) if corner[j] == -25 else self.rngs[e].uniform(0.30, 0.60)
                            for j, e in enumerate(envs)])
            xy = self._points_xy(envs, pidx)
            acts = np.array([self._clip_space(float(xy[j, 0]), float(xy[j, 1]), dx1[j], dy1[j]) for j in range(n)])
            for j, e in enumerate(envs):
                self.init_actions[int(e)].append(acts[j].copy())
            self._step_subset(envs, acts, initialize=True)
            self._update_subset(envs, 500)
        elif self.init_type == "tier3":    # cloth_env.py:951-982
            iters_up = np.array([self.rngs[e].uniform(low=200, high=280) for e in envs])
            lim = 0.25
            acts = np.zeros((n, 4))
            for j, e in enumerate(envs):
                rs = self.rngs[e]
                p0x = _randval_minabs(rs, 0.30, 0.70); p0y = _randval_minabs(rs, 0.30, 0.70)
                dx0 = _randval_minabs(rs, -lim, lim, 0.10); dy0 = _randval_minabs(rs, -lim, lim, 0.10)
                dx0 = _prevent_oob(p0x, dx0); dy0 = _prevent_oob(p0y, dy0)
                acts[j] = self._clip_space(p0x, p0y, dx0, dy0)
                self.init_actions[int(e)].append(acts[j].copy())
            self.reset_iters_up = iters_up
            self._step_subset(envs, acts, initialize=True, iters_up=iters_up)
            self._update_subset(envs, 800)
        else:
            raise ValueError(self.init_type)

    # ------------------------------------------------------------------ step (cloth_env.py:369-534)
    def step(self, actions, host_out=None):
        """One env.step for every environment.

        actions: np.ndarray / sequence [n_env, 4]  -> host decode (bit-exact with CPython), host results
                 torch CUDA tensor [n_env, 4]      -> device decode, results stay on the device
        Returns (obs, reward, done, info) with info = dict of per-env arrays (cloth_env.py:524-533)."""
        c = self.cloth
        if isinstance(actions, torch.Tensor) and actions.is_cuda:
            c.step_actions(actions.to(self.torch_dtype).contiguous())
            obs, rew, done = (c.obs if self.renderer is None else self.image_obs()), c.reward, c.done
            info = self._info(c.coverage, c.variance_inv, c.flags, c.num_steps, c.num_sim_steps)
            return obs, rew, done, info
        a = np.asarray(actions, np.float64).reshape(self.n_env, 4)
        out = host_out if host_out is not None else self.host_buffers()
        c.step_host(a, out)
        info = self._info(out["coverage"], out["variance_inv"], out["flags"], None, None)
        info["sim_steps"] = out["sim_steps"]
        if self.renderer is not None:
            img = self.image_obs()
            if getattr(self, "_host_img", None) is None or self._host_img.shape != img.shape:
                self._host_img = torch.zeros(img.shape, dtype=torch.uint8).pin_memory()
            self._host_img.copy_(img, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            return self._host_img.numpy(), out["reward"], out["done"], info
        return out["obs"], out["reward"], out["done"], info

    def host_buffers(self):
        """Pinned host arrays for step(): reused across calls."""
        if getattr(self, "_host", None) is None:
            n = self.n_env
            npdt = torch.float32 if self.torch_dtype == torch.float32 else torch.float64
            pin = lambda *s, dt: torch.zeros(*s, dtype=dt).pin_memory()
            t = {"obs": pin(n, 3 * self.N, dt=npdt), "reward": pin(n, dt=torch.float64), "done": pin(n, dt=torch.int32),
                 "coverage": pin(n, dt=torch.float64), "variance_inv": pin(n, dt=torch.float64),
                 "flags": pin(n, dt=torch.int32), "sim_steps": pin(n, dt=torch.int32)}
            self._host_t = t
            self._host = {k: v.numpy() for k, v in t.items()}
        return self._host

    def _info(self, coverage, variance_inv, flags, num_steps, num_sim_steps):
        return {"actual_coverage": coverage, "variance_inv": variance_inv,
                "have_tear": (flags & _l.FLAG_TEAR) != 0, "out_of_bounds": (flags & _l.FLAG_OOB) != 0,
                "no_grab": (flags & _l.FLAG_NOGRAB) != 0, "bad_state": (flags & _l.FLAG_BADSTATE) != 0,
                "num_steps": num_steps if num_steps is not None else self.cloth.num_steps,
                "num_sim_steps": num_sim_steps if num_sim_steps is not None else self.cloth.num_sim_steps,
                "start_coverage": self.start_coverage, "start_variance_inv": self.start_variance_inv}

    def get_random_action(self, atype="over_xy_plane"):   # cloth_env.py:989-1018
        if atype == "over_xy_plane":
            return np.stack([self.action_space.sample() for _ in range(self.n_env)])
        if atype == "touch_cloth":
            # the reference supports this only without delta actions (assert at :1006); with them the pick point is a
            # mesh point drawn from np_random as there and (dx, dy) come from the action space
            pidx = np.array([r.randint(self.N) for r in self.rngs])
            xy = self._points_xy(np.arange(self.n_env), pidx)
            a = np.stack([self.action_space.sample() for _ in range(self.n_env)]).astype(np.float64)
            a[:, 0] = (xy[:, 0] - 0.5) * 2; a[:, 1] = (xy[:, 1] - 0.5) * 2
            return a
        raise ValueError(atype)

    # ------------------------------------------------------------------ state pool (fast synthetic resets)
    def snapshot(self):
        c = self.cloth
        return {"pos": c.pos.clone(), "prev": c.prev.clone(), "cov": c.coverage.clone(),
                "rest": None if c.rest is None else c.rest.clone()}

    def reset_from_pool(self, pool, envs, choice):
        """Copy pool states choice[j] into environments envs[j] (device-side, no physics)."""
        c = self.cloth
        e = torch.as_tensor(envs, device=self.device); k = torch.as_tensor(choice, device=self.device)
        c.pos[e] = pool["pos"][k]; c.prev[e] = pool["prev"][k]
        c.prev_coverage[e] = pool["cov"][k]
        self.start_coverage[e] = pool["cov"][k]
        c.flags[e] = 0; c.num_steps[e] = 0; c.num_sim_steps[e] = 0


class _PointView(object):
    """Read/write view of one point of the facade's host copy (point.pyx:17-58 attribute names)."""
    __slots__ = ("_c", "_i")

    def __init__(self, cloth, i):
        self._c, self._i = cloth, i

    x = property(lambda s: float(s._c._host()[0][s._i, 0]))
    y = property(lambda s: float(s._c._host()[0][s._i, 1]))
    z = property(lambda s: float(s._c._host()[0][s._i, 2]))
    px = property(lambda s: float(s._c._host()[1][s._i, 0]))
    py = property(lambda s: float(s._c._host()[1][s._i, 1]))
    pz = property(lambda s: float(s._c._host()[1][s._i, 2]))
    pinned = property(lambda s: bool(s._c._host()[2][s._i]))
    orig_x = property(lambda s: float(s._c._orig[s._i, 0]))
    orig_y = property(lambda s: float(s._c._orig[s._i, 1]))
    orig_z = property(lambda s: float(s._c._orig[s._i, 2]))
    identity_0 = property(lambda s: float(s._i // s._c.width))
    identity_1 = property(lambda s: float(s._i % s._c.width))

    def __repr__(self):
        return "({:.3f}, {:.3f}, {:.3f})".format(self.x, self.y, self.z)


class _ClothFacade(object):
    """`env.cloth`: the names of gym_cloth.physics.cloth.Cloth that callers use (cloth.pyx:390-408, analytic.py:105-125)."""

    def __init__(self, benv):
        self._b = benv
        self.params = benv.cfg
        self.width = benv.P.num_width_points; self.height = benv.P.num_height_points
        self.bounds = (1, 1, 1)
        self._cache = None
        self._orig = None
        self.pts = [_PointView(self, i) for i in range(benv.N)]

    def _invalidate(self):
        self._cache = None

    def _host(self):
        if self._cache is None:
            pos, prev, pin, _ = self._b.cloth.get_state(0)
            self._cache = (pos, prev, pin)
        return self._cache

    @property
    def init_side(self):
        return bool(self._b.init_side[0])

    @property
    def have_tear(self):
        return bool(self._b.cloth.flags[0].item() & _l.FLAG_TEAR)

    @property
    def allpts_arr(self):
        return self._host()[0].copy()

    @property
    def pinnedpts_arr(self):
        pos, _, pin = self._host()
        return pos[pin]

    def update(self):
        self._b.cloth.update(1); self._invalidate()


class _GripperFacade(object):
    """`env.gripper`: gym_cloth.physics.gripper.Gripper (gripper.pyx)."""

    def __init__(self, benv, cloth):
        self._b, self.cloth = benv, cloth
        self.grip_radius = benv.grip_radius

    @property
    def grabbed_pts(self):
        m = self._b.cloth.get_state(0)[3]
        return [self.cloth.pts[i] for i in np.repeat(np.arange(len(m)), m)]

    def grab_top(self, x, y):
        self._b.cloth.grab_top((x, y), self.grip_radius); self.cloth._invalidate()

    def adjust(self, x, y, z):
        self._b.cloth.adjust(x, y, z); self.cloth._invalidate()

    def release(self):
        self._b.cloth.release(); self.cloth._invalidate()


class ClothEnv(object):
    """Drop-in for gym_cloth.envs.ClothEnv on the hot path: same constructor, reset/step/seed/state and the
    attributes scripts read (cloth_env.py:58-186, 332-534, 717-796).  dtype='f64' reproduces the reference
    bit for bit; 'f32' is the production precision."""
    metadata = {"render.modes": ["human"]}

    def __init__(self, cfg_file, subrank=None, start_state_path=None, dtype="f64", device=None):
        self.cfg_file = cfg_file
        self._b = BatchedClothEnv(cfg_file, 1, dtype=dtype, device=device, dom_rand_draws=True)
        self.cfg = self._b.cfg
        env = self.cfg["env"]
        for k in ("max_actions", "iters_up", "iters_up_rest", "iters_pull_max", "iters_grip_rest", "iters_rest",
                  "reduce_factor", "grip_radius"):
            setattr(self, k, env[k])
        self.reward_type = env["reward_type"]
        self.bounds = (1, 1, 1)
        self.render_proc = None
        self._logger_idx = subrank
        self._occlusion_vec = [True, True, True, True]
        self.num_w = self._b.P.num_width_points; self.num_h = self._b.P.num_height_points
        self.num_points = self._b.N
        self.action_space = self._b.action_space
        self.observation_space = self._b.observation_space
        # cloth_env.py:120-124: the reference's {"pts": [Point], "springs": [Spring]} pickle (or the array dict earlier
        # versions of this package wrote)
        self._start_state = None
        if start_state_path is not None:
            self._start_state = self._read_start_state(start_state_path)
        self.cloth = _ClothFacade(self._b)
        self.gripper = _GripperFacade(self._b, self.cloth)
        self.num_steps = 0; self.num_sim_steps = 0; self.have_tear = False
        self._current_coverage = 0.0
        self.seed()

    # the reference reads these from the env, keep them live
    @property
    def np_random(self):
        return self._b.rngs[0]

    def seed(self, seed=None):
        return self._b.seed(seed)

    @property
    def state(self):                       # cloth_env.py:188-209
        if self._b.renderer is not None:
            return self._b.image_obs()[0].cpu().numpy()
        return self.cloth.allpts_arr.reshape(-1)

    def _sync_counters(self):
        c = self._b.cloth
        self.num_steps = int(c.num_steps[0].item()); self.num_sim_steps = int(c.num_sim_steps[0].item())
        self.have_tear = bool(c.flags[0].item() & _l.FLAG_TEAR)

    def _read_start_state(self, path):
        from .. import state_io
        try:
            st = state_io.state_to_arrays(state_io.load_state(path), self._b.P.num_width_points)
        except ValueError:
            with open(path, "rb") as fh:
                st = pickle.load(fh)
            if not (isinstance(st, dict) and "pos" in st and "prev" in st):
                raise
        return st

    def reset(self):
        b = self._b
        if self._start_state is not None:
            # cloth_env.py:736-741: Cloth(state=deepcopy(start_state)) - pts and springs as saved, no init actions
            st = self._start_state
            b.init_side[0] = b.rngs[0].rand() > 0.5      # Cloth.__init__ still draws init_side (cloth.pyx:75)
            b.cloth.set_state(st["pos"], st["prev"], st.get("pinned"))
            if "rest" in st:
                rest = np.nan_to_num(np.asarray(st["rest"], np.float64))
                if rest.size == 6 * b.N:                 # slot order q*6+k (state_io)
                    b.cloth.rest = torch.from_numpy(rest).to(b.device, b.torch_dtype); b.cloth.rest_env_stride = 0
                    b.cloth.exact_rest = True
                else:                                    # spring-list order
                    b.cloth.set_rest(rest)
            b.cloth.num_steps.zero_(); b.cloth.num_sim_steps.zero_()
            b._measure_subset(np.arange(1))
            b.cloth.prev_coverage.copy_(b.cloth.coverage)
            b.start_coverage.copy_(b.cloth.coverage); b.start_variance_inv.copy_(b.cloth.variance_inv)
        else:
            b.reset()
        self.cloth._invalidate()
        if self._start_state is None:
            self.cloth._orig = b.orig_pos[0].cpu().numpy()
        elif "orig" in self._start_state:
            self.cloth._orig = np.array(self._start_state["orig"], np.float64)     # Point.orig_* travel with the pickle
        elif self.cloth._orig is None:
            self.cloth._orig = self.cloth.allpts_arr
        self._sync_counters()
        self._start_coverage = float(b.start_coverage[0].item())
        self._start_variance_inv = float(b.start_variance_inv[0].item())
        self._prev_reward = self._start_coverage
        return self.state

    def step(self, action, initialize=False):
        b = self._b
        a = np.array([float(v) for v in action], np.float64).reshape(1, 4)
        if initialize:
            b._step_subset(np.arange(1), a, initialize=True)
            self.cloth._invalidate()
            return None
        obs, rew, done, info = b.step(a)
        self.cloth._invalidate()
        self._sync_counters()
        self._current_coverage = float(info["actual_coverage"][0])
        self._prev_reward = self._current_coverage
        out_info = {"num_steps": self.num_steps, "num_sim_steps": self.num_sim_steps,
                    "actual_coverage": self._current_coverage, "start_coverage": self._start_coverage,
                    "variance_inv": float(info["variance_inv"][0]), "start_variance_inv": self._start_variance_inv,
                    "have_tear": self.have_tear, "out_of_bounds": bool(info["out_of_bounds"][0])}
        if b.renderer is not None:
            return np.array(obs[0]), float(rew[0]), bool(done[0]), out_info
        return np.array(obs[0], np.float64), float(rew[0]), bool(done[0]), out_info

    def _compute_coverage(self):
        self._b._measure_subset(np.arange(1)); return float(self._b.cloth.coverage[0].item())

    def _compute_variance(self):
        self._b._measure_subset(np.arange(1)); return float(self._b.cloth.variance_inv[0].item())

    def _out_of_bounds(self):
        self._b._measure_subset(np.arange(1)); return bool(self._b.cloth.flags[0].item() & _l.FLAG_OOB)

    def get_random_action(self, atype="over_xy_plane"):
        return self._b.get_random_action(atype)[0]

    def save_state(self, cloth_file):
        """cloth_env.py:343-350: pickle {"pts": cloth.pts, "springs": cloth.springs} - the reference's own object graph
        (gym_cloth_b200/state_io.py), loadable by the reference's ClothEnv(start_state_path=...) and by this one."""
        from .. import state_io
        b = self._b
        pos, prev, pin, _ = b.cloth.get_state(0)
        orig = self.cloth._orig if self.cloth._orig is not None else pos
        state_io.save_state(cloth_file, pos, prev, pin, orig, self._rest_slots(), b.P.num_width_points, self.bounds)

    def _rest_slots(self):
        """Spring.rest_length of environment 0 in slot order q*6+k (double)."""
        import ctypes as C
        c = self._b.cloth
        if c.rest is not None:
            r = c.rest if c.rest_env_stride == 0 else c.rest[0]
            return r.double().cpu().numpy()
        # f32 tier-1/3 batches keep no table: the construction-time lengths of the flat grid (cloth.pyx:417), in double
        N = self._b.N
        pos4 = np.zeros((N, 4)); prev4 = np.zeros((N, 4)); rest6 = np.zeros(6 * N)
        _l.check(_l.lib().clothb200_init_grid_f64(C.byref(self._b.P), 1, None, 1, pos4.ctypes.data, prev4.ctypes.data,
                                                  rest6.ctypes.data), "init_grid")
        return rest6

    def render(self, filepath, mode="human", close=False):
        pass   # the OpenGL viewer is a display-only side channel (SURVEY.md §2 row 12)
