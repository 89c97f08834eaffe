"""BatchedAnts: Python host object over one libantsrl_b200 handle = E independent AntsRL environments on one GPU.

The methods mirror the reference's step-loop surface, batched over a leading env axis:
    observe()            <-> RLApi.observation()    (environment/RL_api.py:96-165)
    step(rot, ph)        <-> RLApi.step()           (environment/RL_api.py:168-204)
    update(noise)        <-> Environment.update()   (environment/environment.py:42-47)
PyTorch is used only as plumbing (device tensors for actions / outputs, the current CUDA stream)."""
import ctypes as C

import numpy as np

from . import _cabi
from ._cabi import AntsConfig, AntsHostState, AntsStats, AntsError, check

DEFAULT_MASK = np.array([[0, 0, 1, 1, 1, 0, 0],
                         [0, 1, 1, 1, 1, 1, 0],
                         [1, 1, 1, 1, 1, 1, 1],
                         [1, 1, 1, 1, 1, 1, 1],
                         [1, 1, 1, 1, 1, 1, 1],
                         [0, 1, 1, 1, 1, 1, 0],
                         [0, 0, 1, 1, 1, 0, 0]], dtype=bool)    # environment_generator.py:35-41

_REWARD_KINDS = {"all": _cabi.REWARD_ALL, "explore": _cabi.REWARD_EXPLORE, "food": _cabi.REWARD_FOOD}
_EVAP_MODES = {"dense": _cabi.EVAP_DENSE, "tiles": _cabi.EVAP_ACTIVE_TILES, "lazy": _cabi.EVAP_LAZY}
KERNEL_FAMILIES = ("move", "food_commit", "perceive", "collide", "rocks", "evaporate", "deposit", "absorb", "misc",
                   "env_move", "env_update", "env_update_move", "pack", "reset")


def make_config(w, h, n_ants, n_phero=2, n_rocks=0, max_time=1000, radius=3, mask="default", fwd_delta=4,
                channels=None, reward_kind="all", reward_factors=(1, 2, 10, 1, 3), reward_threshold=1.0,
                max_speed=1.0, max_rot_speed=40 / 180 * np.pi, carry_speed_reduction=0.05,
                backward_speed_reduction=0.5, diffuse_factor=0.0, evap_factor=0.001, phero_max_val=255.0,
                max_hold=5.0):
    """Environment configuration dict.  Defaults: main.py:42-50, environment_generator.py:35-43,93,97,
    pheromone.py:5-6.  ``channels`` is the perceived_objects list (environment_generator.py:64-99) as names:
    "ants", "phero<k>", "anthill", "walls", "food", "rocks"."""
    if channels is None:
        channels = ["ants"] + ["phero%d" % k for k in range(n_phero)] + ["anthill", "walls", "food"]
        if n_rocks > 0:
            channels.append("rocks")
    if isinstance(mask, str):
        mask = DEFAULT_MASK.copy()
    return dict(w=int(w), h=int(h), n_ants=int(n_ants), n_phero=int(n_phero), n_rocks=int(n_rocks),
                max_time=int(max_time), radius=int(radius), mask=mask, fwd_delta=float(fwd_delta),
                channels=list(channels), reward_kind=reward_kind, reward_factors=tuple(reward_factors),
                reward_threshold=float(reward_threshold), max_speed=float(max_speed),
                max_rot_speed=float(max_rot_speed), carry_speed_reduction=float(carry_speed_reduction),
                backward_speed_reduction=float(backward_speed_reduction), diffuse_factor=float(diffuse_factor),
                evap_factor=float(evap_factor), phero_max_val=phero_max_val, max_hold=float(max_hold))


def _channel_code(name):
    if name == "ants":
        return _cabi.CH_ANTS, 0
    if name.startswith("phero"):
        return _cabi.CH_PHERO, int(name[5:])
    return {"anthill": _cabi.CH_ANTHILL, "walls": _cabi.CH_WALLS, "food": _cabi.CH_FOOD,
            "rocks": _cabi.CH_ROCKS}[name], 0


def build_c_config(cfg, n_envs, device=0, evap_mode="dense", rng_seed=0, env_id_base=0, delta=1.1, record="f64"):
    c = AntsConfig()
    c.abi_version = _cabi.ABI_VERSION
    c.device = int(device)
    c.n_envs, c.n_ants, c.w, c.h = int(n_envs), cfg["n_ants"], cfg["w"], cfg["h"]
    c.n_phero, c.n_rocks, c.max_time = cfg["n_phero"], cfg["n_rocks"], cfg["max_time"]
    c.radius = cfg["radius"]
    s = 2 * cfg["radius"] + 1
    if cfg["mask"] is not None:
        m = np.asarray(cfg["mask"]).astype(bool)
        if m.shape != (s, s):
            raise ValueError("mask shape %r does not match radius %d" % (m.shape, cfg["radius"]))
        c.has_mask = 1
        for k, v in enumerate(m.reshape(-1)):
            c.mask[k] = 1 if v else 0
    else:
        c.has_mask = 0
    if len(cfg["channels"]) > _cabi.MAX_CHANNELS:
        raise ValueError("too many perception channels")
    c.n_channels = len(cfg["channels"])
    for k, name in enumerate(cfg["channels"]):
        c.channel_kind[k], c.channel_arg[k] = _channel_code(name)
    c.delta, c.fwd_delta = float(delta), cfg["fwd_delta"]
    c.reward_threshold, c.max_speed, c.max_rot_speed = cfg["reward_threshold"], cfg["max_speed"], cfg["max_rot_speed"]
    c.carry_speed_reduction, c.backward_speed_reduction = cfg["carry_speed_reduction"], cfg["backward_speed_reduction"]
    c.reward_kind = _REWARD_KINDS[cfg["reward_kind"]]
    rf = list(cfg["reward_factors"]) + [0.0] * 5
    for k in range(5):
        c.reward_factors[k] = float(rf[k])
    c.diffuse_factor, c.evap_factor = cfg["diffuse_factor"], cfg["evap_factor"]
    c.has_max_val = 0 if cfg["phero_max_val"] is None else 1
    c.phero_max_val = 0.0 if cfg["phero_max_val"] is None else float(cfg["phero_max_val"])
    c.max_hold = cfg["max_hold"]
    c.rng_seed, c.env_id_base = int(rng_seed), int(env_id_base)
    c.evap_mode = _EVAP_MODES[evap_mode]
    c.record_format = {"f64": _cabi.REC_F64, "compact": _cabi.REC_COMPACT, "compact8": _cabi.REC_COMPACT8}[record]
    return c


_STATE_F64 = ("x", "y", "theta", "prev_x", "prev_y", "prev_theta", "holding", "seed", "activation",
              "rw_holding_prev", "rw_prev_dist", "rewards", "phero", "food", "anthill_food",
              "rock_centers", "rock_radii", "rock_weights")
_STATE_U8 = ("mandibles", "reward_state", "explored", "walls")


class BatchedAnts:
    def __init__(self, cfg, n_envs, device=0, evap_mode="dense", rng_seed=0, env_id_base=0, use_torch_stream=True,
                 record="f64"):
        import torch
        if not torch.cuda.is_available():
            raise AntsError("antsrl_b200 needs a CUDA device; there is no CPU fallback")
        self._torch = torch
        self.lib = _cabi.load_library()
        self.cfg = dict(cfg)
        self.E, self.N, self.W, self.H = int(n_envs), cfg["n_ants"], cfg["w"], cfg["h"]
        self.P, self.R = cfg["n_phero"], cfg["n_rocks"]
        self.S = 2 * cfg["radius"] + 1
        self.C = len(cfg["channels"])
        self.device = torch.device("cuda", device)
        self.env_id_base = int(env_id_base)          # global id of env 0 (sharding: seeds, Philox streams)
        self._c_cfg = build_c_config(cfg, n_envs, device, evap_mode, rng_seed, env_id_base, record=record)
        h = C.c_void_p()
        check(self.lib, self.lib.ants_create(C.byref(self._c_cfg), C.byref(h)))
        self._h = h
        if use_torch_stream:
            with torch.cuda.device(self.device):
                check(self.lib, self.lib.ants_set_stream(self._h, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        self._out = None
        self._pinned = {}

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            for ptr in self._pinned.values():
                self.lib.ants_host_free(C.c_void_p(ptr[0]))
            self._pinned = {}
            self.lib.ants_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ state
    def _shapes(self, n_envs=None):
        E, N, W, H, P, R = self.E if n_envs is None else n_envs, self.N, self.W, self.H, self.P, self.R
        sh = {k: (E, N) for k in ("x", "y", "theta", "prev_x", "prev_y", "prev_theta", "holding", "seed",
                                  "rw_holding_prev", "rw_prev_dist", "rewards", "mandibles", "reward_state")}
        sh.update(activation=(E, N, P), phero=(E, P, W, H), food=(E, W, H), walls=(E, W, H), explored=(E, W, H),
                  anthill_xyr=(E, 3), anthill_food=(E,), rock_centers=(E, R, 2), rock_radii=(E, R),
                  rock_weights=(E, R))
        return sh

    def import_state(self, state, envs=None):
        """state: dict of numpy arrays with a leading env axis (missing keys are left untouched); scalars
        ``timestep``, ``rw_alias``, ``act_bool`` apply to the whole batch.  With ``envs=(env0, n)`` the arrays hold
        only that window of environments (a new episode for some envs; a large batch uploaded in slices)."""
        env0, n_envs = (0, self.E) if envs is None else (int(envs[0]), int(envs[1]))
        if env0 < 0 or n_envs < 1 or env0 + n_envs > self.E:
            raise ValueError("env window (%d, %d) outside the batch of %d envs" % (env0, n_envs, self.E))
        hs = AntsHostState()
        keep = []
        sh = self._shapes(n_envs)
        for k in _STATE_F64 + _STATE_U8 + ("anthill_xyr",):
            if k not in state or state[k] is None:
                continue
            dt = np.float64 if k in _STATE_F64 else (np.uint8 if k in _STATE_U8 else np.int32)
            a = np.ascontiguousarray(np.asarray(state[k]), dtype=dt)
            if a.shape != sh[k]:
                raise ValueError("state[%r] has shape %r, expected %r" % (k, a.shape, sh[k]))
            if a.size == 0:
                continue
            keep.append(a)
            ptr_t = {np.float64: C.POINTER(C.c_double), np.uint8: C.POINTER(C.c_uint8),
                     np.int32: C.POINTER(C.c_int32)}[dt]
            setattr(hs, k, a.ctypes.data_as(ptr_t))
        # scalars: 0 / -1 = "leave as it is" (a fresh handle starts at timestep 1, aliased reward, bool activations)
        hs.timestep = int(state["timestep"]) if state.get("timestep") is not None else 0
        hs.rw_alias = (1 if state["rw_alias"] else 0) if state.get("rw_alias") is not None else -1
        hs.act_bool = (1 if state["act_bool"] else 0) if state.get("act_bool") is not None else -1
        check(self.lib, self.lib.ants_import_env_state(self._h, env0, n_envs, C.byref(hs)))

    def generate_env_maps(self, anthill_xyr, wall_discs, food_discs, envs=None):
        """ants_generate_env_maps: new maps for all envs, or with ``envs=(env0, n)`` for that window, written on the
        device from the discs of CirclesGenerator maps: anthill_xyr (n, 3), wall_discs (n, Kw, 3), food_discs (n, Kf, 3)
        int arrays of (xc, yc, r).  Pheromones, explored and occupancy are cleared; ants, rocks, the anthill store and
        the batch scalars are left to :meth:`import_state`.

        Either map argument may instead be a :class:`~antsrl_b200.perlin.PerlinLayer` (``PerlinGenerator.layer``: the
        (n, 2) offsets of PerlinGenerator maps and the generator's parameters); that layer is then written from the
        Perlin noise on the device (ants_generate_env_maps_ex), bit for bit as `PerlinGenerator.stamp`."""
        from .perlin import PerlinLayer, perlin_layer_struct
        env0, n_envs = (0, self.E) if envs is None else (int(envs[0]), int(envs[1]))
        hill = np.ascontiguousarray(anthill_xyr, dtype=np.int32)
        keep, layers, discs = [], [], []
        for what, m in (("wall", wall_discs), ("food", food_discs)):
            if isinstance(m, PerlinLayer):
                st, offs = perlin_layer_struct(m)
                if offs.shape[0] != n_envs:
                    raise ValueError("%s layer: expected the offsets of %d envs, got %r" % (what, n_envs, offs.shape))
                keep.append(offs)
                layers.append(C.pointer(st))
                discs.append(np.zeros((n_envs, 0, 3), dtype=np.int32))
            else:
                layers.append(None)
                discs.append(np.ascontiguousarray(m, dtype=np.int32))
        wd, fd = discs
        if hill.shape != (n_envs, 3) or wd.ndim != 3 or wd.shape[0] != n_envs or wd.shape[2] != 3 \
                or fd.ndim != 3 or fd.shape[0] != n_envs or fd.shape[2] != 3:
            raise ValueError("expected anthill_xyr (%d, 3), wall_discs and food_discs (%d, K, 3); got %r, %r, %r"
                             % (n_envs, n_envs, hill.shape, wd.shape, fd.shape))
        i32 = C.POINTER(C.c_int32)
        check(self.lib, self.lib.ants_generate_env_maps_ex(self._h, env0, n_envs, hill.ctypes.data_as(i32),
                                                           int(wd.shape[1]), wd.ctypes.data_as(i32), layers[0],
                                                           int(fd.shape[1]), fd.ctypes.data_as(i32), layers[1]))

    def export_state(self, keys=None, envs=None):
        """The state dict of the whole batch, or with ``envs=(env0, n)`` of that window of environments only
        (arrays then have a leading axis of n) -- what a snapshot of one environment of a large batch needs."""
        env0, n_envs = (0, self.E) if envs is None else (int(envs[0]), int(envs[1]))
        if env0 < 0 or n_envs < 1 or env0 + n_envs > self.E:
            raise ValueError("env window (%d, %d) outside the batch of %d envs" % (env0, n_envs, self.E))
        sh = self._shapes(n_envs)
        hs = AntsHostState()
        out = {}
        for k in _STATE_F64 + _STATE_U8 + ("anthill_xyr",):
            if keys is not None and k not in keys:
                continue
            dt = np.float64 if k in _STATE_F64 else (np.uint8 if k in _STATE_U8 else np.int32)
            a = np.zeros(sh[k], dtype=dt)
            out[k] = a
            if a.size == 0:
                continue
            ptr_t = {np.float64: C.POINTER(C.c_double), np.uint8: C.POINTER(C.c_uint8),
                     np.int32: C.POINTER(C.c_int32)}[dt]
            setattr(hs, k, a.ctypes.data_as(ptr_t))
        check(self.lib, self.lib.ants_export_env_state(self._h, env0, n_envs, C.byref(hs)))
        out["timestep"] = int(hs.timestep)
        out["rw_alias"] = bool(hs.rw_alias)
        out["act_bool"] = bool(hs.act_bool)
        return out

    def activate_all_pheromones(self, new_activations):
        """Ants.activate_all_pheromones (ants.py:86-87) for the whole batch: (E, N, P) array."""
        a = np.asarray(new_activations)
        is_bool = a.dtype == bool
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.shape != (self.E, self.N, self.P):
            raise ValueError("activations must have shape %r" % ((self.E, self.N, self.P),))
        check(self.lib, self.lib.ants_activate_all_pheromones(self._h, a.ctypes.data_as(C.c_void_p), int(is_bool)))

    # ------------------------------------------------------------------ device-resident step loop
    def _buffers(self):
        if self._out is None:
            t = self._torch
            E, N, S, Cn = self.E, self.N, self.S, self.C
            self._out = dict(
                obs=t.empty((E, N, S, S, Cn), dtype=t.float32, device=self.device),
                agent_state=t.empty((E, N, 2), dtype=t.float32, device=self.device),
                state=t.empty((E, N, 2 + self.P), dtype=t.float32, device=self.device),
                reward=t.empty((E, N), dtype=t.float64, device=self.device))
        return self._out

    @staticmethod
    def _ptr(t):
        return C.c_void_p(0 if t is None else t.data_ptr())

    def _check_action(self, a, name):
        if a is None:
            return None
        t = self._torch
        if not (isinstance(a, t.Tensor) and a.is_cuda and a.dtype == t.int8 and a.is_contiguous()
                and tuple(a.shape) == (self.E, self.N)):
            raise ValueError("%s must be a contiguous int8 CUDA tensor of shape (E, N) or None" % name)
        return a

    def observe(self):
        """-> (obs (E,N,S,S,C) f32, agent_state (E,N,2) f32, state (E,N,2+P) f32, reward (E,N) f64), CUDA tensors
        owned by this object and overwritten by the next call."""
        o = self._buffers()
        check(self.lib, self.lib.ants_observe(self._h, self._ptr(o["obs"]), self._ptr(o["agent_state"]),
                                              self._ptr(o["state"]), self._ptr(o["reward"])))
        return o["obs"], o["agent_state"], o["state"], o["reward"]

    def step(self, rotation, pheromone):
        """rotation / pheromone: int8 CUDA tensors (E, N) or None.  -> (obs, agent_state, reward, done)."""
        o = self._buffers()
        rot = self._check_action(rotation, "rotation")
        ph = self._check_action(pheromone, "pheromone")
        done = C.c_int32(0)
        check(self.lib, self.lib.ants_step(self._h, self._ptr(rot), self._ptr(ph), self._ptr(o["obs"]),
                                           self._ptr(o["agent_state"]), self._ptr(o["reward"]), C.byref(done)))
        return o["obs"], o["agent_state"], o["reward"], bool(done.value)

    def update(self, noise=None):
        """noise: f64 CUDA tensor (E, N) of uniforms replacing walls.py:28's draws, or None for Philox."""
        if noise is not None:
            t = self._torch
            if not (isinstance(noise, t.Tensor) and noise.is_cuda and noise.dtype == t.float64
                    and noise.is_contiguous() and tuple(noise.shape) == (self.E, self.N)):
                raise ValueError("noise must be a contiguous float64 CUDA tensor of shape (E, N)")
        check(self.lib, self.lib.ants_update(self._h, self._ptr(noise)))

    def _check_tape(self, a, name, T=None):
        if a is None:
            return None, T
        t = self._torch
        if not (isinstance(a, t.Tensor) and a.is_cuda and a.dtype == t.int8 and a.is_contiguous() and a.dim() == 3
                and tuple(a.shape[1:]) == (self.E, self.N)):
            raise ValueError("%s must be a contiguous int8 CUDA tensor of shape (T, E, N) or None" % name)
        if T is not None and int(a.shape[0]) != T:
            raise ValueError("%s holds %d steps, expected %d" % (name, int(a.shape[0]), T))
        return a, int(a.shape[0])

    def rollout(self, rot_tape, ph_tape, n_steps=None):
        """T x [step; update] with device-resident int8 tapes (T, E, N) (either may be None = the reference's None
        action, then ``n_steps`` gives T) and Philox collision noise; returns the outputs of the last step."""
        o = self._buffers()
        rot, T = self._check_tape(rot_tape, "rot_tape", None if n_steps is None else int(n_steps))
        ph, T = self._check_tape(ph_tape, "ph_tape", T)
        if T is None:
            raise ValueError("rollout without tapes needs n_steps")
        check(self.lib, self.lib.ants_rollout(self._h, self._ptr(rot), self._ptr(ph), T,
                                              self._ptr(o["obs"]), self._ptr(o["agent_state"]), self._ptr(o["reward"])))
        return o["obs"], o["agent_state"], o["reward"]

    def sample_actions(self, seed, n_rotations=3, n_pheromones=3):
        """The agents' exploration branch (collect_agent.py:172-177) drawn on the device: int8 CUDA tensors
        rotation in {-(n//2) .. n - 1 - n//2} and pheromone in {0 .. n_pheromones-1}, shape (E, N)."""
        import torch
        if not hasattr(self, "_act_buf"):
            shape = (self.E, self.N)
            self._act_buf = (torch.empty(shape, dtype=torch.int8, device=self.device),
                             torch.empty(shape, dtype=torch.int8, device=self.device))
        rot, ph = self._act_buf
        check(self.lib, self.lib.ants_sample_actions(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(n_rotations),
                                                     int(n_pheromones), self._ptr(rot), self._ptr(ph)))
        return rot, ph

    # ------------------------------------------------------------------ host-buffer path (numpy in / numpy out)
    def pinned(self, name, shape, dtype):
        """A page-locked numpy array owned by this object (ants_host_alloc)."""
        key = (name, tuple(shape), np.dtype(dtype).str)
        if key not in self._pinned:
            n = int(np.prod(shape)) * np.dtype(dtype).itemsize
            ptr = self.lib.ants_host_alloc(max(n, 1))
            if not ptr:
                raise AntsError("ants_host_alloc failed: %s" % self.lib.ants_last_error().decode())
            buf = (C.c_uint8 * max(n, 1)).from_address(ptr)
            arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
            self._pinned[key] = (ptr, arr)
        return self._pinned[key][1]

    def _host_out(self):
        E, N, S, Cn = self.E, self.N, self.S, self.C
        return (self.pinned("obs", (E, N, S, S, Cn), np.float32), self.pinned("as", (E, N, 2), np.float32),
                self.pinned("state", (E, N, 2 + self.P), np.float32), self.pinned("reward", (E, N), np.float64))

    def observe_host(self):
        obs, ast, st, rw = self._host_out()
        check(self.lib, self.lib.ants_observe_host(self._h, obs.ctypes.data_as(C.c_void_p), ast.ctypes.data_as(C.c_void_p),
                                                   st.ctypes.data_as(C.c_void_p), rw.ctypes.data_as(C.c_void_p)))
        return obs, ast, st, rw

    def step_host(self, rotation, pheromone):
        """numpy int8 (E, N) arrays or None (ideally from :meth:`pinned`); outputs are pinned numpy arrays."""
        obs, ast, _, rw = self._host_out()

        def hp(a):
            if a is None:
                return C.c_void_p(0)
            if not (isinstance(a, np.ndarray) and a.dtype == np.int8 and a.flags.c_contiguous and a.shape == (self.E, self.N)):
                raise ValueError("actions must be contiguous int8 numpy arrays of shape (E, N)")
            return a.ctypes.data_as(C.c_void_p)
        done = C.c_int32(0)
        check(self.lib, self.lib.ants_step_host(self._h, hp(rotation), hp(pheromone), obs.ctypes.data_as(C.c_void_p),
                                                ast.ctypes.data_as(C.c_void_p), rw.ctypes.data_as(C.c_void_p), C.byref(done)))
        return obs, ast, rw, bool(done.value)

    def packed_layout(self):
        """AntsPackedLayout of this handle's observation (include/antsrl_b200.h)."""
        if not hasattr(self, "_layout"):
            L = _cabi.AntsPackedLayout()
            check(self.lib, self.lib.ants_packed_layout(C.byref(self._c_cfg), C.byref(L)))
            self._layout = L
        return self._layout

    def step_host_packed(self, rotation, pheromone):
        """RLApi.step with the observation left in its packed PCIe form on the host (a pinned uint8 array
        (E, N, bytes_per_ant) owned by this object); :meth:`unpack_obs` expands all or part of it."""
        L = self.packed_layout()
        if not L.supported:
            raise AntsError("this configuration has no packed observation form")
        packed = self.pinned("packed", (self.E, self.N, int(L.bytes_per_ant)), np.uint8)
        _, ast, _, rw = self._host_out()

        def hp(a):
            if a is None:
                return C.c_void_p(0)
            if not (isinstance(a, np.ndarray) and a.dtype == np.int8 and a.flags.c_contiguous and a.shape == (self.E, self.N)):
                raise ValueError("actions must be contiguous int8 numpy arrays of shape (E, N)")
            return a.ctypes.data_as(C.c_void_p)
        done = C.c_int32(0)
        check(self.lib, self.lib.ants_step_host_packed(self._h, hp(rotation), hp(pheromone), packed.ctypes.data_as(C.c_void_p),
                                                       ast.ctypes.data_as(C.c_void_p), rw.ctypes.data_as(C.c_void_p), C.byref(done)))
        return packed, ast, rw, bool(done.value)

    def unpack_obs(self, packed, out=None, n_threads=0):
        """packed (..., bytes_per_ant) uint8 -> dense float32 (..., S, S, C), bit-identical to what step_host returns."""
        L = self.packed_layout()
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        n = packed.size // int(L.bytes_per_ant)
        shape = packed.shape[:-1] + (self.S, self.S, self.C)
        if out is None:
            out = np.empty(shape, np.float32)
        check(self.lib, self.lib.ants_unpack_obs(C.byref(L), packed.ctypes.data_as(C.c_void_p), n,
                                                 out.ctypes.data_as(C.c_void_p), int(n_threads)))
        return out

    def update_host(self, noise=None):
        if noise is None:
            check(self.lib, self.lib.ants_update_host(self._h, C.c_void_p(0)))
            return
        a = np.ascontiguousarray(noise, dtype=np.float64)
        if a.shape != (self.E, self.N):
            raise ValueError("noise must have shape (E, N)")
        check(self.lib, self.lib.ants_update_host(self._h, a.ctypes.data_as(C.c_void_p)))

    # ------------------------------------------------------------------ introspection
    def synchronize(self):
        check(self.lib, self.lib.ants_synchronize(self._h))

    def stats(self):
        s = AntsStats()
        check(self.lib, self.lib.ants_get_stats(self._h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in AntsStats._fields_}

    def set_profiling(self, on):
        check(self.lib, self.lib.ants_set_profiling(self._h, int(bool(on))))

    def reset_kernel_ms(self):
        check(self.lib, self.lib.ants_reset_kernel_ms(self._h))

    def kernel_ms(self):
        out = {}
        for name in KERNEL_FAMILIES:
            ms, n = C.c_double(0), C.c_int64(0)
            check(self.lib, self.lib.ants_get_kernel_ms(self._h, name.encode(), C.byref(ms), C.byref(n)))
            out[name] = (ms.value, n.value)
        return out
