"""Host-side map interface: the reference's EnvironmentGenerator / CirclesGenerator semantics
(generator/environment_generator.py:19-106, generator/map_generators.py:28-46) producing plain state dicts that
`BatchedAnts.import_state` uploads.  Runs once per episode on the host; nothing here is on the step path.

Seeding follows the reference exactly (`random.seed(seed); np.random.seed(seed * 5)`, then the same draws in the
same order from the *global* generators), so the same seed yields the same anthill, walls, food, rocks and ants
as the reference, also with user-supplied duck-typed generators that draw from the global RNGs themselves."""
import random

import numpy as np

from .batch import DEFAULT_MASK, make_config


def disc_area(w, h, cx, cy, r):
    """bool (w, h): ((cx - x)^2 + (cy - y)^2)^0.5 <= r on integers -- anthill.py:28-33 without the Python loop
    (exact: all quantities are integers, so the comparison can be done on squares)."""
    xs = np.arange(w, dtype=np.int64)[:, None]
    ys = np.arange(h, dtype=np.int64)[None, :]
    return (cx - xs) ** 2 + (cy - ys) ** 2 <= int(r) * int(r) if r >= 0 else np.zeros((w, h), dtype=bool)


class CirclesGenerator:
    """map_generators.py:28-46: union of n discs; three `random.random()` draws per disc (radius, xc, yc)."""

    def __init__(self, n_circles, min_radius, max_radius):
        self.n_circles = n_circles
        self.min_radius = min_radius
        self.max_radius = max_radius
        self._stamps = {}

    def _stamp(self, r):
        if r not in self._stamps:
            d = np.arange(-r, r + 1, dtype=np.int64)
            self._stamps[r] = d[:, None] ** 2 + d[None, :] ** 2 <= r * r
        return self._stamps[r]

    def draw_discs(self, w, h):
        """-> int32 (n_circles, 3) array of (xc, yc, r): exactly the `random.random()` calls of `generate`, in its order.
        Every disc lies inside the map (xc - r >= 0, xc + r < w, same for y) whenever w, h > 2 * max_radius, up to a
        draw rounding to the upper end; `disc_inside` tells."""
        out = np.empty((self.n_circles, 3), dtype=np.int32)
        for i in range(self.n_circles):
            radius = int(random.random() * (self.max_radius - self.min_radius) + self.min_radius)
            xc = int(random.random() * (w - 2 * radius) + radius)
            yc = int(random.random() * (h - 2 * radius) + radius)
            out[i] = (xc, yc, radius)
        return out

    def stamp(self, w, h, discs):
        """bool (w, h): the union of the discs, with the reference's indexing (gen[x, y] for x in [xc - r, xc + r])."""
        gen = np.zeros((w, h), dtype=bool)
        for xc, yc, radius in np.asarray(discs).tolist():
            xi = np.arange(xc - radius, xc + radius + 1)
            yi = np.arange(yc - radius, yc + radius + 1)
            if xi[0] >= 0 and xi[-1] < w and yi[0] >= 0 and yi[-1] < h:
                gen[xi[0]:xi[-1] + 1, yi[0]:yi[-1] + 1] |= self._stamp(radius)
            else:   # degenerate maps smaller than a disc: same wrap-around / IndexError behaviour as numpy
                st = self._stamp(radius)
                for a, x in enumerate(xi):
                    for b, y in enumerate(yi):
                        if st[a, b]:
                            gen[x, y] = True
        return gen

    def generate(self, w, h):
        return self.stamp(w, h, self.draw_discs(w, h))


def disc_inside(discs, w, h):
    """True iff every (xc, yc, r) disc has r >= 0 and lies inside the w x h map (what ants_generate_env_maps takes)."""
    d = np.asarray(discs, dtype=np.int64).reshape(-1, 3)
    return bool(np.all((d[:, 2] >= 0) & (d[:, 0] - d[:, 2] >= 0) & (d[:, 0] + d[:, 2] < w) &
                       (d[:, 1] - d[:, 2] >= 0) & (d[:, 1] + d[:, 2] < h)))


from .perlin import PerlinGenerator   # noqa: E402,F401  (map_generators.py:9-25; parity unpinned, see perlin.py)


def generate_state(w, h, n_ants, n_pheromones, n_rocks, food_generator, walls_generator, seed=None, max_hold=5,
                   draw_ant_seed=True):
    """environment_generator.py:52-99 -> one env's initial state dict (shared schema, no env axis)."""
    if seed is not None:
        random.seed(seed)
        np.random.seed(seed * 5)
    m = min(w, h)
    ax = int(random.random() * w * 0.5 + w * 0.25)
    ay = int(random.random() * h * 0.5 + h * 0.25)
    ar = int(random.random() * m * 0.05 + m * 0.05)
    area = disc_area(w, h, ax, ay, ar)
    walls = np.asarray(walls_generator.generate(w, h)).copy()
    walls[area] = False
    walls = walls.astype(bool)
    food = np.asarray(food_generator.generate(w, h)).astype(float)
    food *= (1 - walls)
    st = {"walls": walls.astype(np.uint8), "food": food, "anthill_xyr": np.array([ax, ay, ar], dtype=np.int32)}
    if n_rocks > 0:   # environment_generator.py:76-85 with the evident intent `self.n_rocks` (Q17)
        c = np.random.random((n_rocks, 2))
        c[:, 0] *= w * 0.75
        c[:, 1] *= h * 0.25
        c[:, 0] += w * 0.25
        c[:, 1] += h * 0.25
        st["rock_centers"] = c
        st["rock_radii"] = np.random.random(n_rocks) * 5 + 5
        st["rock_weights"] = np.random.random(n_rocks) * 50 + 50
    ang = np.random.random(n_ants) * 2 * np.pi
    dist = np.random.random(n_ants) * ar * 0.8
    x = np.cos(ang) * dist + ax
    y = np.sin(ang) * dist + ay
    t = np.random.random(n_ants) * 2 * np.pi
    st["x"] = np.mod(x, w)                      # Ants.__init__ -> warp_xy, ants.py:28
    st["y"] = np.mod(y, h)
    st["theta"] = t
    if draw_ant_seed:
        st["seed"] = np.random.random(n_ants)   # ants.py:41
    st["activation"] = np.zeros((n_ants, n_pheromones))
    st["act_bool"] = True                       # ants.py:83
    st["rw_alias"] = True
    st["timestep"] = 1
    return st


def stack_states(states, reward_kind="all"):
    """list of per-env dicts -> batched dict with a leading env axis (+ All_Rewards' initial distance)."""
    out = {}
    for k in states[0]:
        if k in ("act_bool", "rw_alias", "timestep"):
            out[k] = states[0][k]
        else:
            out[k] = np.stack([np.asarray(s[k]) for s in states])
    if reward_kind == "all" and "rw_prev_dist" not in out:      # reward_custom.py:77
        out["rw_prev_dist"] = _prev_dist(out["x"], out["y"], out["anthill_xyr"])
    return out


def _prev_dist(x, y, anthill_xyr):
    """All_Rewards' initial distance to the anthill (reward_custom.py:77), the rule of stack_states."""
    ax = np.asarray(anthill_xyr)[..., 0:1].astype(float)
    ay = np.asarray(anthill_xyr)[..., 1:2].astype(float)
    return ((x - ax) ** 2 + (y - ay) ** 2) ** 0.5


def generate_episode(w, h, n_ants, n_pheromones, n_rocks, food_generator, walls_generator, seed=None, max_hold=5,
                     draw_ant_seed=True, perlin=False):
    """The random draws of `generate_state` with the same arguments, from the global RNGs in the same order, without
    the planes: a dict of anthill_xyr (3,), wall_discs / food_discs (n, 3) int32, the rocks, the ants' x, y, theta,
    seed and rw_prev_dist.  -> None when the episode has no disc form (a generator that is not a CirclesGenerator:
    nothing is drawn then; or a disc that does not lie inside the map): `generate_state` builds such maps.

    With ``perlin=True`` a layer whose generator is exactly a `PerlinGenerator` has a draw form too: its two offsets,
    returned as wall_perlin / food_perlin (2,) int32 instead of wall_discs / food_discs."""
    kinds = []
    for g in (walls_generator, food_generator):
        if type(g) is CirclesGenerator:
            kinds.append("discs")
        elif perlin and type(g) is PerlinGenerator:
            kinds.append("perlin")
        else:
            return None
    if seed is not None:
        random.seed(seed)
        np.random.seed(seed * 5)
    m = min(w, h)
    ax = int(random.random() * w * 0.5 + w * 0.25)
    ay = int(random.random() * h * 0.5 + h * 0.25)
    ar = int(random.random() * m * 0.05 + m * 0.05)
    ep = {"anthill_xyr": np.array([ax, ay, ar], dtype=np.int32)}
    for name, g, kind in (("wall", walls_generator, kinds[0]), ("food", food_generator, kinds[1])):   # walls first
        ep[name + "_" + kind] = g.draw_discs(w, h) if kind == "discs" else g.draw_offsets()
    if n_rocks > 0:   # generate_state's draws, same order
        c = np.random.random((n_rocks, 2))
        c[:, 0] *= w * 0.75
        c[:, 1] *= h * 0.25
        c[:, 0] += w * 0.25
        c[:, 1] += h * 0.25
        ep["rock_centers"] = c
        ep["rock_radii"] = np.random.random(n_rocks) * 5 + 5
        ep["rock_weights"] = np.random.random(n_rocks) * 50 + 50
    ang = np.random.random(n_ants) * 2 * np.pi
    dist = np.random.random(n_ants) * ar * 0.8
    x = np.cos(ang) * dist + ax
    y = np.sin(ang) * dist + ay
    t = np.random.random(n_ants) * 2 * np.pi
    ep["x"] = np.mod(x, w)
    ep["y"] = np.mod(y, h)
    ep["theta"] = t
    if draw_ant_seed:
        ep["seed"] = np.random.random(n_ants)
    ep["rw_prev_dist"] = _prev_dist(ep["x"], ep["y"], ep["anthill_xyr"])
    if not all(disc_inside(ep[k], w, h) for k in ("wall_discs", "food_discs") if k in ep):
        return None
    return ep


class BatchedEnvironmentGenerator:
    """E environments, env e generated exactly like the reference generator with seed = seed_base + e."""

    def __init__(self, w, h, n_ants, n_pheromones, n_rocks, food_generator, walls_generator, max_steps,
                 seed_base=1000, perception_mask=None, perception_shift=4, **cfg_kw):
        self.w, self.h, self.n_ants, self.n_pheromones, self.n_rocks = w, h, n_ants, n_pheromones, n_rocks
        self.food_generator, self.walls_generator = food_generator, walls_generator
        self.max_steps, self.seed_base = max_steps, seed_base
        mask = DEFAULT_MASK.copy() if perception_mask is None else np.asarray(perception_mask).astype(bool)
        self.cfg = make_config(w, h, n_ants, n_phero=n_pheromones, n_rocks=n_rocks, max_time=max_steps,
                               radius=mask.shape[0] // 2, mask=mask, fwd_delta=perception_shift, **cfg_kw)

    def generate_states(self, n_envs, first_env=0):
        return [generate_state(self.w, self.h, self.n_ants, self.n_pheromones, self.n_rocks, self.food_generator,
                               self.walls_generator, seed=self.seed_base + first_env + e) for e in range(n_envs)]

    def generate(self, n_envs, device=0, first_env=0, float_activation=True, **batch_kw):
        """-> BatchedAnts holding envs [first_env, first_env + n_envs) (global ids, for sharding).  Defaults to the
        fast field representation the configuration allows: lazy decay and, for one or two pheromones without
        diffusion, the compact 8-byte cell records."""
        from .batch import BatchedAnts
        batch_kw.setdefault("evap_mode", "lazy")
        if self.cfg.get("diffuse_factor", 0.0) == 0.0 and 1 <= self.n_pheromones <= 2 and batch_kw["evap_mode"] == "lazy":
            batch_kw.setdefault("record", "compact8")
        states = self.generate_states(n_envs, first_env)
        batch = BatchedAnts(self.cfg, n_envs, device=device, env_id_base=first_env, **batch_kw)
        batch.import_state(stack_states(states, self.cfg["reward_kind"]))
        if float_activation and self.n_pheromones > 0:   # what agent.initialize does, collect_agent.py:100-102
            batch.activate_all_pheromones(np.ones((n_envs, self.n_ants, self.n_pheromones)) * 10.0)
        return batch

    def reset(self, batch, seed_base, envs=None, float_activation=True, perlin="host"):
        """A new episode for every env of `batch` (a BatchedAnts of this configuration), or with ``envs=(env0, n)`` for
        that window only (main.py:66-79 generates a new environment per episode).  Env e gets the episode drawn with
        seed ``seed_base + batch.env_id_base + e`` (its global id, as in `generate`), and the handle ends up in the state
        `generate` would build from those seeds; a window reset keeps the batch's timestep and flags (lockstep).

        With CirclesGenerator walls and food whose discs all lie inside the map, only the draws are made on the host
        (`generate_episode`) and the maps are written on the device (`BatchedAnts.generate_env_maps`); otherwise (Perlin
        walls, a duck-typed generator, a map smaller than a disc) the complete state is built on the host and imported.
        With ``perlin="device"`` a layer of an exact `PerlinGenerator` takes the device path too: its two offsets are
        drawn on the host and the noise is computed where the records are written, bit for bit as `perlin.py`.  The
        default, ``perlin="host"``, keeps such maps on the host path; making "device" the default (and removing the
        option) is meant to follow once its numbers are measured at scale.  Both paths give the same result.
        -> "device" or "host", the path taken."""
        if perlin not in ("host", "device"):
            raise ValueError("perlin must be 'host' or 'device', not %r" % (perlin,))
        env0, n = (0, batch.E) if envs is None else (int(envs[0]), int(envs[1]))
        if env0 < 0 or n < 1 or env0 + n > batch.E:
            raise ValueError("env window (%d, %d) outside the batch of %d envs" % (env0, n, batch.E))
        seeds = [seed_base + batch.env_id_base + env0 + e for e in range(n)]
        args = (self.w, self.h, self.n_ants, self.n_pheromones, self.n_rocks, self.food_generator, self.walls_generator)
        eps = []
        for s in seeds:
            ep = generate_episode(*args, seed=s, perlin=perlin == "device")
            if ep is None:
                break
            eps.append(ep)
        N, P = self.n_ants, self.n_pheromones
        if len(eps) == n:
            path = "device"
            layers = []
            for name, g in (("wall", self.walls_generator), ("food", self.food_generator)):
                if name + "_perlin" in eps[0]:
                    layers.append(g.layer(np.stack([ep[name + "_perlin"] for ep in eps])))
                else:
                    layers.append(np.stack([ep[name + "_discs"] for ep in eps]))
            batch.generate_env_maps(np.stack([ep["anthill_xyr"] for ep in eps]), layers[0], layers[1], envs=(env0, n))
            keys = ("x", "y", "theta", "seed", "rw_prev_dist") + (("rock_centers", "rock_radii", "rock_weights")
                                                                  if self.n_rocks > 0 else ())
            st = {k: np.stack([ep[k] for ep in eps]) for k in keys}
        else:
            path = "host"
            st = stack_states([generate_state(*args, seed=s) for s in seeds], "all")
            for k in ("act_bool", "rw_alias", "timestep"):
                st.pop(k)
            st["phero"] = np.zeros((n, P, self.w, self.h))
            st["explored"] = np.zeros((n, self.w, self.h), dtype=np.uint8)
        # the per-ant state of a new episode (Ants.__init__, All_Rewards.__init__), the anthill store emptied
        if self.cfg["reward_kind"] != "all":
            st["rw_prev_dist"] = np.zeros((n, N))        # (generate() leaves it as a new handle has it)
        st["prev_x"], st["prev_y"], st["prev_theta"] = st["x"], st["y"], st["theta"]
        for k in ("holding", "rewards", "rw_holding_prev"):
            st[k] = np.zeros((n, N))
        st["mandibles"] = np.zeros((n, N), dtype=np.uint8)
        st["reward_state"] = np.zeros((n, N), dtype=np.uint8)
        st["anthill_food"] = np.zeros(n)
        floats = float_activation and P > 0            # what agent.initialize does, collect_agent.py:100-102
        st["activation"] = np.full((n, N, P), 10.0 if floats else 0.0)
        if n == batch.E:
            st["timestep"], st["rw_alias"], st["act_bool"] = 1, True, not floats
        batch.import_state(st, envs=(env0, n))
        return path
