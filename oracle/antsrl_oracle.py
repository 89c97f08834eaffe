"""CPU oracle for the AntsRL environment step loop -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A numpy restatement of the reference algorithm behind ``RLApi.observation`` / ``RLApi.step`` /
``Environment.update`` (reference: SelennLamson/AntsRL, ``/root/reference``).  Every function cites the
reference file:line it follows.  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import this module, and only as the checker or the timed CPU
baseline -- the product path (``antsrl_b200``) never imports it and has no CPU fallback.

Parity pinning: PINNED.  The reference ships no tests or golden vectors (SURVEY.md section 4), so the
oracle is pinned against outputs of the reference itself, run in the build container by
``tests/golden/make_golden.py`` (which imports the unmodified reference through
``tests/golden/ref_harness.py``) and committed as ``tests/golden/*.npz``; ``tests/test_oracle_golden.py``
replays every fixture through this oracle and demands bit-identical integer state and bit-identical floats
(the oracle uses the same numpy ufuncs in the same order as the reference, so floats agree to the last bit
on the same numpy build; the test tolerates 1e-12 relative to survive a different libm).

State is an explicit structure-of-arrays dict for ONE environment (the shared schema also used by the C ABI):
  x, y, theta, prev_x, prev_y, prev_theta, holding, seed, rw_holding_prev, rw_prev_dist, rewards : (N,) f64
  mandibles, reward_state : (N,) u8        activation : (N,P) f64
  phero : (P,W,H) f64   food : (W,H) f64   walls, explored : (W,H) u8   (index order [x, y] as the reference)
  anthill_xyr : (3,) i32   anthill_food : f64   rock_centers (R,2), rock_radii (R,), rock_weights (R,) f64
  timestep : int   rw_alias : bool (reward's holding snapshot still aliases the live array, quirk Q18)
  act_bool : bool (phero_activation still has the bool dtype of ants.py:83, so "256" deposits 1.0)
"""
import numpy as np
from scipy.signal import convolve2d

AX = np.newaxis
DELTA = 1.1                 # RL_api.py:15

DEFAULT_MASK = np.array([[0, 0, 1, 1, 1, 0, 0],
                         [0, 1, 1, 1, 1, 1, 0],
                         [1, 1, 1, 1, 1, 1, 1],
                         [1, 1, 1, 1, 1, 1, 1],
                         [1, 1, 1, 1, 1, 1, 1],
                         [0, 1, 1, 1, 1, 1, 0],
                         [0, 0, 1, 1, 1, 0, 0]], dtype=bool)   # environment_generator.py:35-41


def make_config(w, h, n_ants, n_phero=2, n_rocks=0, max_time=1000, radius=3, mask="default", fwd_delta=4,
                channels=None, reward_kind="all", reward_factors=(1, 2, 10, 1, 3), reward_threshold=1.0,
                max_speed=1.0, max_rot_speed=40 / 180 * np.pi, carry_speed_reduction=0.05,
                backward_speed_reduction=0.5, diffuse_factor=0.0, evap_factor=0.001, phero_max_val=255.0,
                max_hold=5.0):
    """Defaults are main.py:42-50 (RLApi / All_Rewards), environment_generator.py:35-43,93,97 and
    pheromone.py:5-6."""
    if channels is None:   # perceived_objects order built by environment_generator.py:64-99
        channels = ["ants"] + ["phero%d" % p for p in range(n_phero)] + ["anthill", "walls", "food"]
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


def diffuse_filter(diffuse_factor, evap_factor):
    """pheromone.py:5-10."""
    f = np.ones((3, 3)) * diffuse_factor
    f[1, 1] = 1 - 8 * diffuse_factor
    f *= 1 - evap_factor
    return f


def anthill_area(w, h, ax, ay, ar):
    """anthill.py:28-33: area[x,y] = ((ax-x)^2 + (ay-y)^2)^0.5 <= r on integers."""
    xs = np.arange(w)[:, AX]
    ys = np.arange(h)[AX, :]
    return ((ax - xs) ** 2 + (ay - ys) ** 2) ** 0.5 <= ar


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; Random123): ten rounds of
    (c0, c1, c2, c3) <- (hi(M1*c2) ^ c1 ^ k0, lo(M1*c2), hi(M0*c0) ^ c3 ^ k1, lo(M0*c0)), the key bumped by the Weyl
    constants after each round.  Counter words are uint64 arrays holding 32-bit values, the key two Python ints."""
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    W0, W1 = 0x9E3779B9, 0xBB67AE85
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = M0 * c0
        p1 = M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0)), lo1, (hi0 ^ c3 ^ np.uint64(k1)), lo0
        k0 = (k0 + W0) & 0xFFFFFFFF
        k1 = (k1 + W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def _ant_counters(seed, env_id, step, n_ants, stream):
    c0 = np.arange(n_ants, dtype=np.uint64)
    c1 = np.full(n_ants, step & 0xFFFFFFFF, dtype=np.uint64)
    c2 = np.full(n_ants, env_id & 0xFFFFFFFF, dtype=np.uint64)
    c3 = np.full(n_ants, stream, dtype=np.uint64)
    return philox4x32_10(c0, c1, c2, c3, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)


def philox_uniform(seed, env_id, step, n_ants):
    """Counter-based collision noise used by the CUDA path in throughput mode (no reference analogue: the
    reference draws from the global numpy RNG, walls.py:28).  Philox4x32-10, counter = (ant, step, env_id, 0),
    key = (seed_lo, seed_hi); u = ((r0 >> 5) * 2^26 + (r1 >> 6)) / 2^53."""
    r0, r1, _, _ = _ant_counters(seed, env_id, step, n_ants, 0)
    a = (r0 >> np.uint64(5)).astype(np.float64)
    b = (r1 >> np.uint64(6)).astype(np.float64)
    return (a * 67108864.0 + b) / 9007199254740992.0


def philox_actions(seed, env_id, step, n_ants, n_rot=3, n_ph=3):
    """Mirror of the CUDA path's on-device action sampler (ants_sample_actions; the agents' exploration branch,
    collect_agent.py:172-177): Philox4x32-10, counter (ant, step, env_id, 1), value = (r * n) >> 32."""
    r0, r1, _, _ = _ant_counters(seed, env_id, step, n_ants, 1)
    rot = ((r0 * np.uint64(n_rot)) >> np.uint64(32)).astype(np.int64) - n_rot // 2
    ph = ((r1 * np.uint64(n_ph)) >> np.uint64(32)).astype(np.int64)
    return rot, ph


class OracleEnv:
    """One environment.  ``cfg`` from :func:`make_config`, ``state`` in the shared schema."""

    def __init__(self, cfg, state):
        self.cfg = cfg
        st = {}
        for k, v in state.items():
            st[k] = np.array(v, copy=True) if isinstance(v, np.ndarray) else v
        n, w, h = cfg["n_ants"], cfg["w"], cfg["h"]
        st.setdefault("prev_x", st["x"].copy()); st.setdefault("prev_y", st["y"].copy())
        st.setdefault("prev_theta", st["theta"].copy())
        st.setdefault("holding", np.zeros(n)); st.setdefault("mandibles", np.zeros(n, np.uint8))
        st.setdefault("reward_state", np.zeros(n, np.uint8))
        st.setdefault("activation", np.zeros((n, cfg["n_phero"])))
        # ants.py:83 makes phero_activation a BOOL array; activate_all_pheromones (ants.py:86-87) replaces it
        # by whatever the caller passes (float in collect_agent.py:101).  While it is bool, the 256 written
        # by activate_pheromone (ants.py:94-96) is stored as True and deposits 1.0.
        st.setdefault("act_bool", True)
        st.setdefault("phero", np.zeros((cfg["n_phero"], w, h)))
        st.setdefault("explored", np.zeros((w, h), np.uint8))
        st.setdefault("anthill_food", np.float64(0.0))
        st.setdefault("timestep", 1)                     # environment.py:27
        st.setdefault("rewards", np.zeros(n))
        st.setdefault("rw_holding_prev", np.zeros(n))
        st.setdefault("rw_alias", True)                  # reward_custom.py:35,66-67 (Q18)
        st.setdefault("rock_centers", np.zeros((0, 2))); st.setdefault("rock_radii", np.zeros(0))
        st.setdefault("rock_weights", np.zeros(0))
        ax, ay, ar = [int(v) for v in st["anthill_xyr"]]
        self.area = anthill_area(w, h, ax, ay, ar)
        if "rw_prev_dist" not in st:                     # reward_custom.py:77 (All_Rewards.setup only)
            st["rw_prev_dist"] = (((st["x"] - ax) ** 2 + (st["y"] - ay) ** 2) ** 0.5
                                  if cfg["reward_kind"] == "all" else np.zeros(n))
        self.s = st
        r = cfg["radius"]
        # RL_api.py:92-93
        self.perception_coords = np.dstack([np.arange(-r, r + 1)[AX, :].repeat(2 * r + 1, 0),
                                            np.arange(-r, r + 1)[:, AX].repeat(2 * r + 1, 1)]).astype(float)
        self.perception_coords *= DELTA
        self.filter = diffuse_filter(cfg["diffuse_factor"], cfg["evap_factor"])

    # ------------------------------------------------------------------ observation (RL_api.py:96-165)
    def sample_points(self):
        """Sample coordinates (N,S,S,2) of every ant before rounding, RL_api.py:100-116."""
        s, cfg = self.s, self.cfg
        xy = np.stack([s["x"], s["y"]], axis=1)
        theta = s["theta"]
        xy_f = xy.copy()
        t_f = theta + np.pi * 0.5
        if cfg["fwd_delta"] != 0:
            xy_f += np.array([np.cos(theta), np.sin(theta)]).T * cfg["fwd_delta"]
        cos_t = np.cos(t_f)
        sin_t = np.sin(t_f)
        rel = self.perception_coords[AX, :, :].repeat(len(theta), 0)
        rx = cos_t[:, AX, AX] * rel[:, :, :, 0] - sin_t[:, AX, AX] * rel[:, :, :, 1]
        ry = sin_t[:, AX, AX] * rel[:, :, :, 0] + cos_t[:, AX, AX] * rel[:, :, :, 1]
        rel[:, :, :, 0], rel[:, :, :, 1] = rx, ry
        return rel + xy_f[:, AX, AX, :]

    def sample_cells(self):
        """Integer sample coordinates (N,S,S,2) of every ant, RL_api.py:100-119."""
        cfg = self.cfg
        ab = np.round(self.sample_points()).astype(int)  # half-to-even, Q11
        ab[:, :, :, 0] = np.mod(ab[:, :, :, 0], cfg["w"])
        ab[:, :, :, 1] = np.mod(ab[:, :, :, 1], cfg["h"])
        return ab

    def observation(self):
        """RL_api.py:96-165.  Returns (perception (N,S,S,C) f64, agent_state (N,2), state (N,2+P)).
        Side effect: reward state (Q8)."""
        s, cfg = self.s, self.cfg
        w, h = cfg["w"], cfg["h"]
        ab = self.sample_cells()
        cx, cy = ab[:, :, :, 0], ab[:, :, :, 1]
        perception = np.zeros(list(ab.shape[:-1]) + [len(cfg["channels"])])
        for i, ch in enumerate(cfg["channels"]):
            if ch.startswith("phero"):                   # :124-125
                perception[:, :, :, i] = s["phero"][int(ch[5:])][cx, cy] / cfg["phero_max_val"]
            elif ch == "food":                           # :126-127
                perception[:, :, :, i] = s["food"][cx, cy]
            elif ch == "walls":                          # :128-129
                perception[:, :, :, i] = s["walls"].astype(bool)[cx, cy]
            elif ch == "anthill":                        # :130-131
                perception[:, :, :, i] = self.area[cx, cy]
            elif ch == "rocks":                          # :132-135 (strict <, Q13)
                vecs = ab[:, :, :, AX, :] - s["rock_centers"][AX, AX, AX, :, :]
                dists = np.sum(vecs ** 2, axis=4) ** 0.5
                perception[:, :, :, i] = np.max(dists < s["rock_radii"], axis=3)
            elif ch == "ants":                           # :136-142 (0/1 occupancy, Q1)
                axy = np.stack([s["x"], s["y"]], axis=1).astype(int)
                axy[:, 0] = np.mod(axy[:, 0], w)
                axy[:, 1] = np.mod(axy[:, 1], h)
                amap = np.zeros((w, h), dtype=int)
                amap[axy[:, 0], axy[:, 1]] += 1
                perception[:, :, :, i] = amap[cx, cy]
            else:
                raise ValueError(ch)
        if cfg["mask"] is not None:                      # :147-148
            perception = np.asarray(cfg["mask"], dtype=bool)[AX, :, :, AX] * (perception + 1) - 1
        n = cfg["n_ants"]
        state = np.zeros((n, 2 + cfg["n_phero"]))        # :155-158
        state[:, 0] = s["mandibles"]
        state[:, 1] = s["holding"]
        state[:, 2:] = s["activation"] > 0
        agent_state = np.zeros((n, 2))                   # :160-162
        agent_state[:, 0] = s["holding"]
        agent_state[:, 1] = s["seed"]
        self._reward_observation(ab, agent_state)        # :164
        return perception, agent_state, state

    def _reward_observation(self, ab, agent_state):
        s, cfg = self.s, self.cfg
        kind = cfg["reward_kind"]
        cx, cy = ab[:, :, :, 0], ab[:, :, :, 1]
        explored = s["explored"].view(bool) if s["explored"].dtype == np.uint8 else s["explored"]
        holding_now = agent_state[:, 0]
        holding_prev = s["holding"] if s["rw_alias"] else s["rw_holding_prev"]   # Q18 aliasing
        if kind == "explore":                            # reward_custom.py:17-22
            s["rewards"] = np.sum(1 - explored[cx, cy], axis=(1, 2)) / 10
            explored[cx, cy] = True
        elif kind == "food":                             # reward_custom.py:37-40
            r = holding_now - holding_prev
            r[r < 0] = 10
            s["rewards"] = r
            s["rw_holding_prev"] = holding_now.copy(); s["rw_alias"] = False
        elif kind == "all":                              # reward_custom.py:79-106
            f_explore, f_food, f_anthill, f_explore_hold, f_heading = cfg["reward_factors"]
            rewards = np.zeros(cfg["n_ants"])
            r_food = holding_now - holding_prev
            r_anthill = r_food.copy()
            r_food[r_food < 0] = 0
            s["rw_holding_prev"] = holding_now.copy(); s["rw_alias"] = False
            if f_explore != 0 or f_explore_hold != 0:
                r_exp = np.sum(1 - explored[cx, cy], axis=(1, 2)) / 10
                r_exp = np.where(holding_now == 0, r_exp * f_explore, r_exp * f_explore_hold)
                explored[cx, cy] = True                  # gather-then-scatter, Q7
                rewards += r_exp
            r_anthill[r_anthill > 0] = 0
            r_anthill[r_anthill < 0] = 1
            ax, ay = int(s["anthill_xyr"][0]), int(s["anthill_xyr"][1])
            new_dist = ((s["x"] - ax) ** 2 + (s["y"] - ay) ** 2) ** 0.5
            heading = (s["rw_prev_dist"] > new_dist) * (s["holding"] > 0) * 0.1
            s["rw_prev_dist"] = new_dist
            rewards += r_food * f_food + r_anthill * f_anthill + heading * f_heading
            s["rewards"] = rewards
        else:
            raise ValueError(kind)

    # ------------------------------------------------------------------ step (RL_api.py:168-204)
    def step(self, rotation, pheromone):
        """rotation, pheromone: (N,) int arrays or None.  Returns (perception, agent_state, reward, done)."""
        s, cfg = self.s, self.cfg
        w, h = cfg["w"], cfg["h"]
        pxy = np.stack([s["prev_x"], s["prev_y"]], axis=1).astype(int)            # :178
        m = s["mandibles"].astype(np.int64)
        for ch in cfg["channels"]:                                                # :180-184 (list order, Q5)
            if ch == "food":
                m = np.bitwise_or(s["food"][pxy[:, 0], pxy[:, 1]] > 0, m)
            elif ch == "anthill":
                m = np.bitwise_and(1 - self.area[s["x"].astype(int), s["y"].astype(int)], m)
        # update_mandibles, ants.py:102-117
        old = s["mandibles"].astype(np.int64)
        closing = np.bitwise_and(m, 1 - old)
        opening = np.bitwise_and(1 - m, old)
        s["mandibles"] = m.astype(np.uint8)
        taken = np.minimum(cfg["max_hold"], np.maximum(0, s["food"][pxy[:, 0], pxy[:, 1]])) * closing
        dropped = s["holding"].copy() * opening
        s["food"][pxy[:, 0], pxy[:, 1]] += dropped - taken                        # last ant wins, Q1
        s["holding"] = s["holding"] + (taken - dropped)
        if pheromone is not None:                                                 # ants.py:89-96 (P == 2)
            ph = np.asarray(pheromone)
            if cfg["n_phero"] != 2:
                raise ValueError("activate_pheromone hard-codes two pheromones (ants.py:92-96)")
            on = 1.0 if s["act_bool"] else 256.0
            act = np.zeros((cfg["n_ants"], 2))
            act[ph == 1, 0] = on
            act[(ph != 0) & (ph != 1), 1] = on
            s["activation"] = act
        if rotation is not None:                                                  # ants.py:62-67
            s["theta"] = np.mod(s["theta"] + np.asarray(rotation) * cfg["max_rot_speed"], 2 * np.pi)
        fwd = np.ones(cfg["n_ants"]) * cfg["max_speed"] * (1 - s["holding"] * cfg["carry_speed_reduction"])
        fwd[fwd < 0] *= cfg["backward_speed_reduction"]                           # :194-195
        s["x"] = np.mod(s["x"] + np.cos(s["theta"]) * fwd, w)                     # ants.py:69-80
        s["y"] = np.mod(s["y"] + np.sin(s["theta"]) * fwd, h)
        perception, agent_state, _ = self.observation()                           # :198 (before collisions, Q2)
        done = cfg["max_time"] == int(s["timestep"])                              # :200 (Q15)
        reward = s["rewards"]                                                     # reward.py:38
        add = ((reward - cfg["reward_threshold"]) > 0) * 255                      # ants.py:119-121
        s["reward_state"] = np.minimum(s["reward_state"].astype(np.int64) + add, 255).astype(np.uint8)
        return perception, agent_state, reward, bool(done)

    # ------------------------------------------------------------------ update (environment.py:42-47)
    def update(self, noise=None):
        """One Environment.update() in the order of SURVEY section 3.4.  ``noise``: (N,) uniforms in [0,1), one per
        ant; only colliding ants consume theirs (walls.py:28 draws one value per hit in ant order)."""
        s, cfg = self.s, self.cfg
        w, h = cfg["w"], cfg["h"]
        s["timestep"] = int(s["timestep"]) + 1                                    # environment.py:45
        walls = s["walls"].astype(bool)
        # 1. Walls (order -1), walls.py:22-30
        cx, cy = s["x"].astype(int), s["y"].astype(int)
        hit = walls[cx, cy]
        if hit.any():
            if noise is None:
                raise ValueError("collision noise required")
            s["x"] = np.where(hit, s["prev_x"], s["x"])
            s["y"] = np.where(hit, s["prev_y"], s["y"])
            th = s["theta"].copy()
            th[hit] += np.asarray(noise, dtype=float)[hit] - 0.5                  # theta not re-wrapped, Q3
            s["theta"] = th
        for p in range(cfg["n_phero"]):
            s["phero"][p][walls] = 0
        # 3. CircleObstacles (order 0), circle_obstacles.py:32-58
        if cfg["n_rocks"] > 0:
            c, rad, wt = s["rock_centers"], s["rock_radii"], s["rock_weights"]
            xy = np.stack([s["x"], s["y"]], axis=1)
            v = c[AX, :, :] - xy[:, AX, :]
            d = np.sum(v ** 2, axis=2) ** 0.5
            push = v * (1 - rad[AX, :] / (d + 0.001))[:, :, AX]
            push[d > rad[AX, :], :] = 0
            c = c - np.sum(push, axis=0) / wt[:, AX]
            s["rock_centers"] = c
            v = c[AX, :, :] - xy[:, AX, :]
            d = np.sum(v ** 2, axis=2) ** 0.5
            push = v * (1 - rad[AX, :] / (d + 0.001))[:, :, AX]
            push[d > rad[AX, :], :] = 0
            xy = xy + np.sum(push, axis=1)
            s["x"] = np.mod(xy[:, 0], w)
            s["y"] = np.mod(xy[:, 1], h)
        # 4. Pheromone (order 0), pheromone.py:43-45
        for p in range(cfg["n_phero"]):
            ph = convolve2d(s["phero"][p], self.filter, 'same', 'fill', 0)
            ph[ph < 0.01] = 0
            s["phero"][p] = ph
        # 6. Ants (order 999), ants.py:123-130 + pheromone.py:36-41
        s["prev_x"], s["prev_y"], s["prev_theta"] = s["x"].copy(), s["y"].copy(), s["theta"].copy()
        cx, cy = s["x"].astype(int), s["y"].astype(int)
        for p in range(cfg["n_phero"]):
            if cfg["n_ants"] > 0:
                s["phero"][p][cx, cy] += s["activation"][:, p]                    # last ant wins, Q1
                if cfg["phero_max_val"] is not None:
                    s["phero"][p] = np.minimum(s["phero"][p], cfg["phero_max_val"])
        s["reward_state"] = (s["reward_state"] * 0.9).astype(np.uint8)            # Q16
        # 7. Anthill (order 1000), anthill.py:41-46
        gain = s["food"] * self.area
        s["food"] -= gain
        s["anthill_food"] = np.float64(s["anthill_food"] + np.sum(gain))

    def activate_all_pheromones(self, new_activations):
        """ants.py:86-87."""
        a = np.asarray(new_activations)
        self.s["act_bool"] = bool(a.dtype == bool)
        self.s["activation"] = a.astype(float).reshape(self.cfg["n_ants"], self.cfg["n_phero"]).copy()

    def export(self):
        out = {}
        for k, v in self.s.items():
            out[k] = np.array(v, copy=True) if isinstance(v, np.ndarray) else v
        return out
