"""Pheromone field kernels at their edges: hand-built fields against the oracle.

The third part of every update -- Walls.update's zeroing of the field, Pheromone.update's convolution and `< 0.01`
cut and the clamp of add_pheromones -- runs in k_diffuse_tma / k_plane_walls (DIFFUSE_FACTOR != 0), k_evaporate_dense
and k_tiles_compact + k_evaporate_tiles (eager fields) or in the lazy decode (plain_value, k_lazy_fold).  Random
scenarios reach their edges only by chance; `field_world` builds one env's complete state that reaches them on
purpose (the ants stand still: no step runs, the updates only deposit):
  * diffusion with the taps ring 1/32 and centre 1/4 (diffuse_factor 1/16, evap_factor 1/2) and every input on a
    2^-10 grid, so that every product and sum is exact in any order: the field must equal scipy's bit for bit.  Unit
    impulses in the corners, on both sides of every 64-cell tile seam of the stencil and at W - 1 / H - 1; impulses
    whose ring or centre product lands one grid step either side of 0.01; walls under, beside and along the seams and
    map edges, some holding pheromone; values at and above max_val; deposits onto wall and non-wall cells; maps of one
    cell width, around the 16-cell padding and across several stencil tiles, P = 1 ... 4;
  * eager fields: values whose product with the centre tap is the largest double below 0.01 or exactly 0.01 (the
    cut's ties, found by walking the doubles), one double either side; tiles that retire and are reactivated, across
    the env boundaries of the compaction's warps, the generic P != 2 branch, windowed imports and resets;
  * the lazy decode: plain values that cross the cut at update 1, 5, 300 (across the 8-bit timestamp folds) and 4100
    (across the 12-bit fold of the f64 records).
The CPU tests replay every batch on the oracle's own arithmetic and assert that each class occurs and that the dyadic
diffusion runs are exact; the GPU tests compare the exported field (bit for bit where the arithmetic is exact), every
observation and the whole state after every call.  With diffusion a negative or NaN activation or imported value is
refused (the sign bit of a plane value is the wall flag)."""
from collections import Counter

import numpy as np
import pytest
from scipy.signal import convolve2d

from oracle.antsrl_oracle import OracleEnv, make_config
from parity_util import compare_state, stack_init
from test_gpu_perception_edges import check_outputs

G = 2.0 ** -10                                  # the grid of every diffusion input
CUT = 0.01
SEAM = 64                                       # k_diffuse_tma's output tile (kStX = kStY)
TILE = 16                                       # the activity tiles of ACTIVE_TILES
DIFFUSE = dict(diffuse_factor=1 / 16, evap_factor=1 / 2)
EXACT_UPDATES, DIFFUSE_UPDATES = 8, 12
NOISE = 0.5                                     # collision noise: theta += 0.5 - 0.5 (an ant standing in a wall)


def field_cfg(w, h, n_phero, n_ants, **kw):
    return make_config(w, h, n_ants, n_phero=n_phero, fwd_delta=0, max_speed=0.0, max_time=100000, **kw)


def below(v):
    return float(np.nextafter(v, -np.inf))


def above(v):
    return float(np.nextafter(v, np.inf))


def preimage(target, c):
    """x with fl(x * c) == target, the doubles around target / c walked outward; None if there is none."""
    lo = hi = target / c
    for _ in range(64):
        for x in (lo, hi):
            if x * c == target:
                return float(x)
        lo, hi = below(lo), above(hi)
    return None


# ------------------------------------------------------------------------------------------------ the worlds
def _seams(n):
    return [s for t in range(SEAM, n, SEAM) for s in (t - 1, t)]


def _diffuse_design(cfg, e):
    """(phero, walls, ant cells, activations) of a diffusion world."""
    W, H, P, N = cfg["w"], cfg["h"], cfg["n_phero"], cfg["n_ants"]
    phero = np.zeros((P, W, H))
    walls = np.zeros((W, H), bool)

    def put(k, x, y, v):
        if 0 <= x < W and 0 <= y < H:
            phero[k, x, y] = v

    def wall(x, y):
        if 0 <= x < W and 0 <= y < H:
            walls[x, y] = True

    for k in range(P):
        s = 1.0 + 0.25 * ((e * P + k) % 7)             # a different field in every env and plane
        y0, x0 = (3 + 2 * e + k) % H, (5 + 2 * e + k) % W
        for x, y in ((0, 0), (W - 1, 0), (0, H - 1), (W - 1, H - 1), (W - 1, y0), (x0, H - 1)):
            put(k, x, y, s)
        for x in _seams(W):
            put(k, x, y0, s)
        for y in _seams(H):
            put(k, x0, y, s)
        # isolated impulses: ring products 327/32 G < 0.01 < 328/32 G, centre products 40/4 G < 0.01 < 41/4 G
        for j, v in enumerate((327, 328, 40, 41)):
            put(k, (W // 2 + 4 * j + 2 * k) % W, (H // 3 + 3 * e) % H, v * G)
        if min(W, H) >= 17:                            # the clamp: a block of 600 (centre output 300), 255 and 300
            bx, by = W // 3, (2 * H) // 3
            for dx in (-1, 0, 1):
                for dy in (-1, 0, 1):
                    put(k, bx + dx, by + dy, 600.0)
            put(k, bx + 5, by, 255.0)
            put(k, bx, by - 5, 300.0)
    for t in range(SEAM, W, SEAM):                     # walls under and beside the seams
        for y in range(H // 4, H // 4 + 6):
            wall(t - 1, y)
            wall(t, y + 7)
            wall(t - 3, y)
    for t in range(SEAM, H, SEAM):
        for x in range(W // 4, W // 4 + 6):
            wall(x, t - 1)
            wall(x + 7, t)
            wall(x, t + 2)
    for j in range(4):                                 # along the map edges, and in a corner
        wall(0, H // 2 + j)
        wall(W - 1, H // 2 + j)
        wall(W // 2 + j, 0)
        wall(W // 2 + j, H - 1)
    wall(W - 1, H - 1)
    for x in _seams(W)[:1]:                            # under a seam impulse
        wall(x, (3 + 2 * e) % H)
    # the ants: one on a wall cell, one on the 255 cell (a deposit of 200 keeps it clamped), the rest free
    rng = np.random.RandomState(700 + e)
    free = [(x, y) for x in range(W) for y in range(H) if not walls[x, y]]
    order = sorted(range(len(free)), key=lambda i: (phero[:, free[i][0], free[i][1]].any(), rng.random_sample()))
    cells = [free[i] for i in order[:N - 1]]
    wl = np.argwhere(walls)
    cells.append(tuple(wl[e % len(wl)]))
    if min(W, H) >= 17:
        cells[0] = (W // 3 + 5, (2 * H) // 3)
    act = np.zeros((N, P))
    small = (0.5 + 37 * G, 41 * G, 2.0 + 5 * G, 0.0)
    for j in range(N):
        for k in range(P):
            act[j, k] = small[(j + k + e) % len(small)]
    if min(W, H) >= 17:
        act[0, :] = 200.0 + 3 * G
    return phero, walls, cells, act


def _ties(c):
    """Values whose first evaporation product is 0.01 -/+ one or two doubles, and their preimages (the tie at the
    second update); the ties themselves are largest-below and exactly 0.01."""
    out = []
    for tgt in (below(below(CUT)), below(CUT), CUT, above(CUT)):
        v = preimage(tgt, c)
        assert v is not None, "no double x with x * %r == %r" % (c, tgt)
        out.append(v)
        v2 = preimage(v, c)
        if v2 is not None:
            out.append(v2)
    return out


def _tiles(W, H):
    return [(tx, ty) for tx in range(-(-W // TILE)) for ty in range(-(-H // TILE))]


def _eager_design(cfg, e):
    """(phero, walls, ant cells, activations) of an eager world: ties, walls holding pheromone, values above max_val;
    tile A holds one value cut at update 1 and an ant that deposits at update 2 (retired, then reactivated), tile B
    one value cut at update 1 and an ant that deposits at update 1; `schedule` below switches their activations."""
    W, H, P, N = cfg["w"], cfg["h"], cfg["n_phero"], cfg["n_ants"]
    c = 1.0 - cfg["evap_factor"]
    phero = np.zeros((P, W, H))
    walls = np.zeros((W, H), bool)
    tiles = _tiles(W, H)
    nt = len(tiles)
    ta, tb, tg, th = (tiles[(e + j) % nt] for j in range(4))
    k0 = e % P
    cut1 = preimage(below(CUT), c)

    def cell(t, dx, dy):
        return min(t[0] * TILE + dx, W - 1), min(t[1] * TILE + dy, H - 1)

    phero[(k0,) + cell(ta, 3, 5)] = cut1
    phero[(k0,) + cell(tb, 2, 9)] = cut1
    ties = _ties(c)
    for j, v in enumerate(ties):
        for k in range(P):
            phero[(k,) + cell(tg, (j * 3 + k) % TILE, (j * 5 + 2 * k) % TILE)] = v
    for j, v in enumerate((255.0, 300.0, 1000.0, 254.9, 0.5)):
        phero[((j + e) % P,) + cell(th, (2 * j + 1) % TILE, (3 * j + 7) % TILE)] = v
    for dx, dy in ((1, 1), (4, 12), (12, 4)):             # walls holding pheromone
        x, y = cell(th, dx, dy)
        walls[x, y] = True
        phero[:, x, y] = 3.5 + e
    cells = [cell(ta, 7, 2), cell(tb, 11, 13)]
    rng = np.random.RandomState(900 + e)
    while len(cells) < N:
        x, y = rng.randint(W), rng.randint(H)
        if (x, y) not in cells and not walls[x, y] and (x // TILE, y // TILE) not in (ta, tb):
            cells.append((x, y))
    act = np.zeros((N, P))
    act[0, k0] = act[1, k0] = 0.0125
    for j in range(2, N):
        act[j, (j + e) % P] = (0.75, 300.0, 0.0)[j % 3]
    return phero, walls, cells, act


def field_world(cfg, e):
    """One env's complete state (OracleEnv / stack_init schema): the diffusion design when diffuse_factor != 0, else
    the eager one.  Ants stand still on distinct cells (max_speed 0, no step runs)."""
    design = _diffuse_design if cfg["diffuse_factor"] != 0.0 else _eager_design
    phero, walls, cells, act = design(cfg, e)
    W, H, N = cfg["w"], cfg["h"], cfg["n_ants"]
    assert len(set(cells)) == N
    x = np.array([cx + 0.375 for cx, _ in cells])
    y = np.array([cy + 0.625 for _, cy in cells])
    return {"x": x, "y": y, "theta": 0.25 + 0.5 * np.arange(N), "holding": np.zeros(N),
            "mandibles": np.zeros(N, np.uint8), "reward_state": np.zeros(N, np.uint8),
            "seed": np.linspace(0.0, 1.0, N), "activation": act, "rw_holding_prev": np.zeros(N),
            "rewards": np.zeros(N), "walls": walls.astype(np.uint8), "food": np.zeros((W, H)), "phero": phero,
            "explored": np.zeros((W, H), np.uint8), "anthill_xyr": np.array([W // 2, H // 2, 0], np.int32),
            "anthill_food": np.float64(0.0), "act_bool": False}


def schedule(cfg, worlds, t):
    """The activations of update t (1-based): eager worlds switch ant 0 (tile A) on at update 2 only and ant 1
    (tile B) on at update 1 only; diffusion worlds keep theirs."""
    act = np.stack([w["activation"] for w in worlds]).copy()
    if cfg["diffuse_factor"] == 0.0:
        if t != 2:
            act[:, 0] = 0.0
        if t != 1:
            act[:, 1] = 0.0
    return act


# ------------------------------------------------------------------------------------------------ batches
# (W, H, P, E): one-cell-wide maps, sizes around the 16-cell padding and the 64-cell stencil tiles, P = 1 ... 4
DIFFUSE_SHAPES = [(1, 70, 1, 3), (70, 1, 2, 3), (2, 3, 3, 3), (17, 15, 4, 4), (63, 64, 1, 3), (64, 63, 2, 3),
                  (65, 65, 3, 4), (64, 128, 4, 3), (129, 127, 2, 4), (130, 67, 3, 5), (200, 260, 1, 3)]


def diffuse_batch(w, h, P, E):
    cfg = field_cfg(w, h, P, 2 if w * h < 20 else 6, **DIFFUSE)
    return cfg, [field_world(cfg, e) for e in range(E)]


# (W, H, P, evap_factor): partial edge tiles, the P == 2 vector branch of k_evaporate_tiles and the generic one
EAGER_SHAPES = [(37, 21, 1, 0.001), (21, 37, 2, 0.001), (45, 19, 3, 0.3), (19, 45, 4, 0.3), (40, 33, 2, 0.3)]
EAGER_E, EAGER_UPDATES = 41, 8


def eager_batch(w, h, P, evap):
    cfg = field_cfg(w, h, P, 5, evap_factor=evap)
    return cfg, [field_world(cfg, e) for e in range(EAGER_E)]


# ------------------------------------------------------------------------------------------------ the oracle
def zero_tiles(cfg, phero):
    """(tiles_x, tiles_y) bool: no non-zero value in any plane of the 16 x 16 tile."""
    W, H = cfg["w"], cfg["h"]
    tx, ty = -(-W // TILE), -(-H // TILE)
    pad = np.zeros((phero.shape[0], tx * TILE, ty * TILE))
    pad[:, :W, :H] = phero != 0.0
    return ~pad.reshape(-1, tx, TILE, ty, TILE).any(axis=(0, 2, 4))


class FieldOracle(OracleEnv):
    """OracleEnv whose update also records the convolution before the cut (`pre`) and the field between the cut and
    the deposits (`evap`), and counts the classes this file builds in `ev`."""

    def __init__(self, cfg, state):
        super().__init__(cfg, state)
        self.ev = Counter()
        self.history = [zero_tiles(cfg, self.s["phero"])]      # zero tiles after each update (and the import)
        self.evap_zero = []

    def update(self, noise=None):
        s, cfg, ev = self.s, self.cfg, self.ev
        walls = s["walls"].astype(bool)
        ph = s["phero"].copy()
        ev["wall_holding"] += int((ph[:, walls] != 0).sum())
        if cfg["phero_max_val"] is not None:
            ev["above_max"] += int((ph > cfg["phero_max_val"]).sum())
        ph[:, walls] = 0
        pre = np.stack([convolve2d(p, self.filter, 'same', 'fill', 0) for p in ph])
        step = 2.0 ** -15 if cfg["diffuse_factor"] != 0.0 else 0.0
        if step:
            ev["cut_step_below"] += int(((pre < CUT) & (pre >= CUT - step)).sum())
            ev["cut_step_above"] += int(((pre >= CUT) & (pre < CUT + step)).sum())
        else:
            ev["tie_below"] += int((pre == below(CUT)).sum())
            ev["tie_at"] += int((pre == CUT).sum())
            ev["double_below_tie"] += int((pre == below(below(CUT))).sum())
            ev["double_above_tie"] += int((pre == above(CUT)).sum())
        evap = np.where(pre < CUT, 0.0, pre)
        if cfg["n_ants"] > 0 and cfg["phero_max_val"] is not None:
            evap = np.minimum(evap, cfg["phero_max_val"])
        ez = zero_tiles(cfg, evap)
        self.evap_zero.append(ez)
        super().update(noise)
        z = zero_tiles(cfg, s["phero"])
        was = ~self.history[-1]
        ev["tile_cut_and_deposit"] += int((was & ez & ~z).sum())
        if len(self.evap_zero) >= 2:
            retired = ~self.history[-2] & self.evap_zero[-2] & self.history[-1]
            ev["tile_retired_reactivated"] += int((retired & ~z).sum())
        self.history.append(z)


def alt_update(cfg, phero, walls, cells, act):
    """The field part of one update in another summation order: centre tap first, then the ring in reverse
    order, neighbours added pairwise."""
    W, H = cfg["w"], cfg["h"]
    f = phero.copy()
    f[:, walls] = 0
    pad = np.zeros((f.shape[0], W + 2, H + 2))
    pad[:, 1:-1, 1:-1] = f
    ring = 1.0 * cfg["diffuse_factor"] * (1 - cfg["evap_factor"])
    centre = (1 - 8.0 * cfg["diffuse_factor"]) * (1 - cfg["evap_factor"])
    nb = [pad[:, 1 + dx:W + 1 + dx, 1 + dy:H + 1 + dy] for dx in (1, 0, -1) for dy in (1, 0, -1) if dx or dy]
    s = ((nb[0] + nb[1]) + (nb[2] + nb[3])) + ((nb[4] + nb[5]) + (nb[6] + nb[7]))
    out = f * centre + s * ring
    out[out < CUT] = 0
    for j, (x, y) in enumerate(cells):
        out[:, x, y] += act[j]
    return np.minimum(out, cfg["phero_max_val"])


def replay(cfg, worlds, T):
    """import; T x [activate (schedule); update] on FieldOracle; the summed class counts and the oracles."""
    oracles = [FieldOracle(cfg, w) for w in worlds]
    for t in range(1, T + 1):
        act = schedule(cfg, worlds, t)
        for e, o in enumerate(oracles):
            o.activate_all_pheromones(act[e])
            o.update(np.full(cfg["n_ants"], NOISE))
    ev = Counter()
    for o in oracles:
        ev.update(o.ev)
    return ev, oracles


def seam_impulses(cfg, worlds):
    n = 0
    for w in worlds:
        ph = w["phero"]
        for t in range(SEAM, cfg["w"], SEAM):
            n += int((ph[:, t - 1] != 0).any() and (ph[:, t] != 0).any())
        for t in range(SEAM, cfg["h"], SEAM):
            n += int((ph[:, :, t - 1] != 0).any() and (ph[:, :, t] != 0).any())
    return n


def test_field_worlds_cover_every_class():
    total = Counter()
    for shape in DIFFUSE_SHAPES:
        cfg, worlds = diffuse_batch(*shape)
        ev, _ = replay(cfg, worlds, 2)
        ev["seam_impulse"] = seam_impulses(cfg, worlds)
        total.update(ev)
    for shape in EAGER_SHAPES:
        cfg, worlds = eager_batch(*shape)
        ev, _ = replay(cfg, worlds, 4)
        for k in ("tie_below", "tie_at", "double_below_tie", "double_above_tie", "tile_retired_reactivated",
                  "tile_cut_and_deposit", "wall_holding", "above_max"):
            assert ev[k] > 0, "%r: no %s; counts %r" % (shape, k, dict(ev))
        total.update(ev)
    for k in ("seam_impulse", "cut_step_below", "cut_step_above", "wall_holding", "above_max"):
        assert total[k] > 0, "no %s; counts %r" % (k, dict(total))
    # lazy: with |delta| < evap_factor a value below the cut is zeroed at update k, one above it at k + 1 (the deltas of
    # 1e-2 cross some updates away: far from the band on both sides)
    evap = LAZY_CFG["evap_factor"]
    crossing = [(k, d) for k, d, ref in lazy_reference(LAZY_CFG)
                if ref[k - 1] > 0 and (ref[k] == 0 if d < 0 else ref[k] > 0 and ref[k + 1] == 0)]
    for k in LAZY_KS:
        for d in LAZY_DELTAS:
            if 1e-11 <= abs(d) < evap:
                assert (k, d) in crossing, "k = %d, delta = %g: the reference does not cross the cut at k" % (k, d)
    print(len(crossing), "of", len(LAZY_KS) * len(LAZY_DELTAS), "lazy cases cross the cut at k exactly")
    print(dict(total))


@pytest.mark.parametrize("shape", DIFFUSE_SHAPES, ids=["%dx%d_P%d" % s[:3] for s in DIFFUSE_SHAPES])
def test_dyadic_diffusion_is_exact(shape):
    """The oracle (scipy's order) and alt_update (another order) agree bit for bit for EXACT_UPDATES updates: every
    product and sum of these runs is exact, so the CUDA stencil's order must give the same bits."""
    cfg, worlds = diffuse_batch(*shape)
    for e, w in enumerate(worlds):
        o = OracleEnv(cfg, w)
        walls = w["walls"].astype(bool)
        cells = [(int(x), int(y)) for x, y in zip(w["x"], w["y"])]
        f = w["phero"].copy()
        for t in range(1, EXACT_UPDATES + 1):
            o.update(np.full(cfg["n_ants"], NOISE))
            f = alt_update(cfg, f, walls, cells, w["activation"])
            assert np.array_equal(o.s["phero"], f), "%r env %d: summation orders differ at update %d" % (shape, e, t)


# ------------------------------------------------------------------------------------------------ lazy plain values
LAZY_KS = (1, 5, 300, 4100)
LAZY_DELTAS = tuple(s * d for d in (1e-2, 1e-5, 1e-8, 1e-11, 1e-14) for s in (1, -1))
LAZY_CFG = field_cfg(24, 18, 2, 4)


def lazy_cases(cfg):
    """(k, delta, v, env, plane, x, y): v = 0.01 / c^k (1 + delta), every case on a cell of its own."""
    c = 1.0 - cfg["evap_factor"]
    out = []
    j = 0
    for k in LAZY_KS:
        for d in LAZY_DELTAS:
            e, p = j % 2, (j // 2) % 2
            out.append((k, d, CUT / c ** k * (1 + d), e, p, 2 + (j // 4) % 20, 2 + 3 * (j // 80) + (j // 4) // 20))
            j += 1
    return out


def lazy_reference(cfg):
    """(k, delta, ref) with ref[t] the reference's value after t updates (pheromone.py:44-45 with DIFFUSE_FACTOR 0:
    one product by the centre tap, then the cut), t = 0 ... max(k) + 1."""
    c = 1.0 - cfg["evap_factor"]
    cases = lazy_cases(cfg)
    v = np.array([cs[2] for cs in cases])
    refs = [v.copy()]
    for _ in range(max(LAZY_KS) + 1):
        v = v * c
        v[v < CUT] = 0.0
        refs.append(v.copy())
    refs = np.array(refs)
    return [(cs[0], cs[1], refs[:, j]) for j, cs in enumerate(cases)]


def lazy_worlds(cfg):
    W, H, N = cfg["w"], cfg["h"], cfg["n_ants"]
    worlds = []
    for e in range(2):
        ph = np.zeros((2, W, H))
        for k, d, v, ce, p, x, y in lazy_cases(cfg):
            if ce == e:
                ph[p, x, y] = v
        worlds.append({"x": np.array([20.5, 21.5, 22.5, 23.5]), "y": np.full(N, 16.5), "theta": np.zeros(N),
                       "seed": np.zeros(N), "activation": np.zeros((N, 2)), "walls": np.zeros((W, H), np.uint8),
                       "food": np.zeros((W, H)), "phero": ph, "explored": np.zeros((W, H), np.uint8),
                       "anthill_xyr": np.array([22, 1, 0], np.int32), "act_bool": False})
    return worlds


# ------------------------------------------------------------------------------------------------ GPU
class FieldPair:
    """A BatchedAnts batch and one OracleEnv per env, driven by imports, activations and updates only; the field and
    the observation compared after every call."""

    def __init__(self, cfg, worlds, evap_mode):
        from antsrl_b200 import BatchedAnts
        import torch
        self.torch, self.cfg, self.worlds = torch, cfg, worlds
        self.E = len(worlds)
        self.o = [OracleEnv(cfg, w) for w in worlds]
        self.b = BatchedAnts(cfg, self.E, evap_mode=evap_mode, record="f64")
        self.b.import_state(stack_init(cfg, worlds))
        self.t = 0
        self.check("import", exact=True)

    def close(self):
        self.b.close()

    def field(self):
        return np.stack([o.s["phero"] for o in self.o])

    def check(self, what, exact):
        st = self.b.export_state()
        compare_state(st, self.o, what, self.cfg)
        ref = self.field()
        if exact:
            bad = np.argwhere(st["phero"] != ref)
            assert bad.size == 0, "%s: the field differs at %d entries, first (env, plane, x, y) %r: %r vs %r" % (
                what, len(bad), tuple(bad[0]), st["phero"][tuple(bad[0])], ref[tuple(bad[0])])
        else:
            np.testing.assert_allclose(st["phero"], ref, rtol=1e-12, atol=0, err_msg=what + ": field")

    def observe(self, what):
        obs, ast, st, rew = self.b.observe()
        refs = []
        for o in self.o:
            p_, a_, s_ = o.observation()
            refs.append((p_, a_, o.s["rewards"].copy(), s_))
        check_outputs(self.cfg, (obs, ast, rew, st), refs, what)

    def update(self, exact):
        self.t += 1
        act = schedule(self.cfg, self.worlds, self.t)
        for o, a in zip(self.o, act):
            o.activate_all_pheromones(a)
        self.b.activate_all_pheromones(act)
        for o in self.o:
            o.update(np.full(self.cfg["n_ants"], NOISE))
        self.b.update(self.torch.full((self.E, self.cfg["n_ants"]), NOISE, dtype=self.torch.float64, device="cuda"))
        self.check("update %d" % self.t, exact)


def run_diffusion(cfg, worlds, evap_mode="dense", hooks=None):
    pr = FieldPair(cfg, worlds, evap_mode)
    try:
        pr.observe("observe after the import")
        for t in range(1, DIFFUSE_UPDATES + 1):
            if hooks and t in hooks:
                hooks[t](pr)
            pr.update(exact=t <= EXACT_UPDATES)
            pr.observe("observe after update %d" % t)
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", DIFFUSE_SHAPES, ids=["%dx%d_P%d" % s[:3] for s in DIFFUSE_SHAPES])
def test_diffusion_stencil_edges(shape):
    """k_diffuse_tma, k_plane_walls, plane deposits, export and the row perception kernel on the dyadic worlds: the
    field bit for bit for EXACT_UPDATES updates, then within 1e-12."""
    run_diffusion(*diffuse_batch(*shape))


@pytest.mark.gpu
def test_diffusion_generic_perception(monkeypatch):
    monkeypatch.setenv("ANTS_PERCEIVE_GENERIC", "1")
    run_diffusion(*diffuse_batch(65, 65, 3, 4), evap_mode="tiles")


def replace_window(pr, env0, worlds):
    """A windowed import of new worlds into envs [env0, env0 + len(worlds))."""
    st = stack_init(pr.cfg, worlds)
    for k in ("act_bool", "rw_alias", "timestep"):
        st.pop(k, None)
    pr.b.import_state(st, envs=(env0, len(worlds)))
    ts = int(pr.o[0].s["timestep"])
    for j, w in enumerate(worlds):
        o = OracleEnv(pr.cfg, dict(w, rw_prev_dist=st["rw_prev_dist"][j]))
        o.s["timestep"], o.s["rw_alias"] = ts, pr.o[env0].s["rw_alias"]
        pr.o[env0 + j] = o
        pr.worlds[env0 + j] = w
    pr.check("after the import of envs [%d, %d)" % (env0, env0 + len(worlds)), exact=True)


def reset_window(pr, env0, n):
    """ants_generate_env_maps for envs [env0, env0 + n): one wall disc, no food; the oracles take the new maps."""
    W, H = pr.cfg["w"], pr.cfg["h"]
    hill = np.array([[W // 2, H // 2, 0]] * n, np.int32)
    pr.b.generate_env_maps(hill, np.array([[[W // 5, H // 5, 2]]] * n, np.int32), np.zeros((n, 0, 3), np.int32),
                           envs=(env0, n))
    keys = ("food", "walls", "phero", "explored", "anthill_xyr")
    maps = pr.b.export_state(keys=keys, envs=(env0, n))
    for j in range(n):
        for k in keys:
            pr.o[env0 + j].s[k] = maps[k][j].copy()
        assert not maps["phero"][j].any()
    pr.check("after the reset of envs [%d, %d)" % (env0, env0 + n), exact=True)


@pytest.mark.gpu
def test_diffusion_window_import_and_reset_on_the_second_plane():
    """A windowed import after 3 updates and a windowed reset after 5: the current planes are then the second half of
    the ping-pong allocation, which k_pack_f64, k_plane_walls and k_reset_maps must write."""
    cfg, worlds = diffuse_batch(130, 67, 3, 5)
    hooks = {4: lambda pr: replace_window(pr, 1, [field_world(cfg, 20 + e) for e in range(2)]),
             6: lambda pr: reset_window(pr, 3, 1)}
    run_diffusion(cfg, worlds, hooks=hooks)


def diffusion_handle(E=2):
    from antsrl_b200 import BatchedAnts
    cfg, worlds = diffuse_batch(17, 15, 2, E)
    b = BatchedAnts(cfg, E, evap_mode="dense", record="f64")
    b.import_state(stack_init(cfg, worlds))
    return cfg, worlds, b


@pytest.mark.gpu
@pytest.mark.parametrize("bad", (-3.0, float("nan")))
def test_diffusion_refuses_negative_values(bad):
    """With diffusion the sign bit of a plane value is the wall flag, so a negative (or NaN) deposit or imported value
    would turn its cell into a wall of the stencil.  activate_all_pheromones and import_state refuse them; a refused
    activate_all_pheromones leaves the handle unchanged."""
    import torch
    from antsrl_b200 import AntsError
    cfg, worlds, b = diffusion_handle()
    try:
        before = b.export_state()
        act = np.stack([w["activation"] for w in worlds])
        act[1, 2, 1] = bad
        with pytest.raises(AntsError):
            b.activate_all_pheromones(act)
        after = b.export_state()
        for k, v in before.items():
            assert np.array_equal(np.asarray(v), np.asarray(after[k])), "refused activations changed %s" % k
        with pytest.raises(AntsError):
            b.import_state({"activation": act})
        ph = np.stack([w["phero"] for w in worlds])
        ph[0, 1, 3, 4] = bad
        with pytest.raises(AntsError):
            b.import_state({"phero": ph})
        with pytest.raises(AntsError):
            b.import_state({"phero": ph[:1]}, envs=(0, 1))
        # the window imported again: the handle runs on as the oracle
        b.import_state(stack_init(cfg, worlds))
        oracles = [OracleEnv(cfg, w) for w in worlds]
        noise = np.full((len(worlds), cfg["n_ants"]), NOISE)
        for o, n in zip(oracles, noise):
            o.update(n)
        b.update(torch.from_numpy(noise).cuda())
        compare_state(b.export_state(), oracles, "after the import that followed the refused ones", cfg)
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("dense", "tiles"))
@pytest.mark.parametrize("shape", EAGER_SHAPES, ids=["%dx%d_P%d_evap%g" % s for s in EAGER_SHAPES])
def test_eager_field_edges(shape, mode):
    """k_evaporate_dense / k_tiles_compact + k_evaporate_tiles: the field bit for bit after every update, through a
    windowed import (envs 10 ... 14) and a windowed reset (envs 20 ... 22) in the middle of the batch; with tiles the
    active_tiles statistic of update k equals the oracle's non-zero tiles after update k - 1."""
    cfg, worlds = eager_batch(*shape)
    pr = FieldPair(cfg, worlds, mode)
    try:
        pr.observe("observe after the import")
        for t in range(1, EAGER_UPDATES + 1):
            if t == 3:
                replace_window(pr, 10, [field_world(cfg, 100 + e) for e in range(5)])
            if t == 5:
                reset_window(pr, 20, 3)
            listed = sum(int((~zero_tiles(cfg, o.s["phero"])).sum()) for o in pr.o)
            pr.update(exact=True)
            if mode == "tiles":
                assert pr.b.stats()["active_tiles"] == listed, "update %d: %d tiles listed, %d hold pheromone" % (
                    t, pr.b.stats()["active_tiles"], listed)
            pr.observe("observe after update %d" % t)
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("record", ("f64", "compact", "compact8"))
def test_lazy_plain_values_at_the_cut(record):
    """Plain values that cross the cut at update k (k = 1, 5, 300, 4100), decoded as v 2^(k log2 c) from f64 or f32
    storage.  The zero / non-zero decision at k and k + 1 may differ from the reference only inside the format's band
    around 0.01 (1e-11 relative for f64 records, (1 + folds) 2^-24 for the f32 ones, DESIGN.md section 4); outside it
    the value is within 1e-12 (f64) or 1e-5."""
    from antsrl_b200 import BatchedAnts
    cfg = LAZY_CFG
    c = 1.0 - cfg["evap_factor"]
    ref = lazy_reference(cfg)
    cases = lazy_cases(cfg)
    bar = 1e-12 if record == "f64" else 1e-5
    b = BatchedAnts(cfg, 2, evap_mode="lazy", record=record)
    agree = {}
    try:
        b.import_state(stack_init(cfg, lazy_worlds(cfg)))
        checkpoints = sorted({t for k in LAZY_KS for t in (k, k + 1)})
        for t in range(1, max(checkpoints) + 1):
            b.update(None)
            if t not in checkpoints:
                continue
            ph = b.export_state(keys=("phero",))["phero"]
            for (k, d, r), (_, _, _, e, p, x, y) in zip(ref, cases):
                g, want = ph[e, p, x, y], r[t]
                pre = r[t - 1] * c                      # the reference's value before its cut at update t
                folds = t // 254 + 1
                band = 1e-11 if record == "f64" else (1 + folds) * 2.0 ** -24
                if t in (k, k + 1):
                    agree[(k, d)] = agree.get((k, d), True) and (g == 0) == (want == 0)
                if abs(pre / CUT - 1) <= band:
                    continue
                assert (g == 0) == (want == 0), "%s, update %d, k %d, delta %g: %r vs the reference's %r" % (
                    record, t, k, d, g, want)
                assert abs(g - want) <= bar * want, "%s, update %d, k %d, delta %g: %r vs %r" % (record, t, k, d, g, want)
    finally:
        b.close()
    for (k, d), ok in agree.items():
        if abs(d) >= 1e-5 or (record == "f64" and abs(d) >= 1e-11):
            assert ok, "%s: k %d, delta %g: the cut decision differs from the reference" % (record, k, d)
