"""Perception kernels at their edges: hand-built worlds against the oracle.

Random scenarios reach the branches and arithmetic tricks of the perception kernels only by chance.  `edge_world`
builds states that reach them on purpose:
  * exact .5 ties of the sample coordinates (np.round is half to even, Q11; ants_perceive_rows.cuh round_half_even),
    in the centre column (X = 0), off it, and below zero (-0.5 -> 0, -1.5 -> W - 2);
  * ants on the seams (0, 1e-9, W - 1e-9 and W itself, Q14) and in every corner, with large headings (Q3);
  * walls, a seam-crossing anthill, several ants on one cell, every class of food record (integer, escaped to the
    side array, 0xFFFF itself), plain pheromone values (below the 0.01 cut, max_val), pre-explored cells and windows
    that share unexplored cells (gather-then-scatter, Q7);
  * rocks: integer centre and radius (samples exactly at the radius read 0, strict <, Q13), a window three rocks
    reach (the further candidates of the row kernel), rocks one cell from a seam (rocks are not on the torus, Q4)
    and 64 rocks (the last bit of the candidate masks).
The CPU test proves on the oracle's own arithmetic that every class occurs and that no sample lies within 1e-12 of a
half without being exactly on it (a 1-ulp libm difference could flip such a near-tie).  The GPU tests run the worlds
through every instance of the row kernel, the generic kernel (also with the window sizes, masks and channel lists the
row kernel never serves, and on maps below the single-wrap threshold) and grouped rollouts whose group ranges start
at ants that leave the observation's bulk store misaligned."""
import numpy as np
import pytest

from oracle.antsrl_oracle import DELTA, OracleEnv, make_config, philox_uniform
from parity_util import compare_state, stack_init

DOWN = -np.pi / 2                      # theta + pi/2 == 0 exactly: cos = 1, sin = 0 in any libm
FOOD_CLASSES = (0.0, 1.0, 0.25, 65534.0, 65535.0, 65536.0, 65536.5)
PHERO_VALUES = (0.005, 0.5, 3.7, 100.0, 255.0)         # 0.005: below the 0.01 cut; 255: max_val
SEAM_THETAS = (DOWN, 0.3, 2.0, 1000.123, -999.77)
NEAR_TIE = 1e-12


def reach_of(cfg):
    """How far a sample lies from its ant, as ants_create bounds it (ants_abi.cu, perceive_slow_wrap): maps no larger
    than this take the generic kernel's slow wrap."""
    return cfg["radius"] * DELTA * 1.5 + abs(cfg["fwd_delta"]) + 2.0


def offsets(radius):
    return np.arange(-radius, radius + 1).astype(float) * DELTA       # RL_api.py:92-93, as the oracle computes them


def disc_mask(radius):
    k = np.arange(-radius, radius + 1)
    return (k[:, None] ** 2 + k[None, :] ** 2) <= radius * radius + radius


def edge_cfg(n_ants, w=40, h=35, radius=3, n_rocks=0, mask="default", channels=None, reward_kind="all"):
    if isinstance(mask, str) and radius != 3:
        mask = disc_mask(radius)
    return make_config(w, h, n_ants, n_phero=2, n_rocks=n_rocks, radius=radius, mask=mask, fwd_delta=0,
                       max_speed=0.0, channels=channels, reward_kind=reward_kind, max_time=1000)


def tie_coord(target, off):
    """x with x + off == target exactly in f64 (the search walks the doubles around target - off)."""
    x0 = target - off
    lo = hi = x0
    for _ in range(256):
        for x in (lo, hi):
            if x + off == target:
                return float(x)
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
    raise AssertionError("no double x with x + %r == %r" % (off, target))


def _sites(cfg):
    """The ant placements (x, y, theta) every world draws its ants from, in a fixed order: neighbours in the list
    (several ants on one cell) tend to land in the same env."""
    W, H, r = cfg["w"], cfg["h"], cfg["radius"]
    off = offsets(r)
    gx, gy = W // 2 + 0.37, H // 2 + 0.37          # fractions 0.37 +- 0.1 k: never near a half
    sites = []

    def ties(n, target_hi):
        """coordinates on an axis of size n whose window has exact ties: X = 0 (even and odd n), X != 0 on both sides,
        below zero and at the far seam"""
        out = [2 * (n // 4) + 0.5, 2 * (n // 4) + 1.5,
               tie_coord(2 * (n // 3) + 0.5, off[r + 1]), tie_coord(2 * (n // 3) + 1.5, off[0]),
               tie_coord(-0.5, off[0]), tie_coord(-1.5, off[0]), tie_coord(-0.5, off[r - 1]),
               tie_coord(n - 0.5, off[-1]), tie_coord(n + 0.5, off[-1]), tie_coord(n + 1.5, off[-1])]
        return [v for v in out if 0.0 <= v < n]
    for x in ties(W, W):
        sites.append((x, gy, DOWN))
    for y in ties(H, H):
        sites.append((gx, y, DOWN))
    sites.append((tie_coord(2 * (W // 3) + 0.5, off[r + 1]), tie_coord(-0.5, off[0]), DOWN))      # both axes
    # several ants on one cell
    cx, cy = 3 * W // 4, H // 4
    sites += [(cx + 0.12, cy + 0.23, 0.3), (cx + 0.63, cy + 0.77, DOWN), (cx + 0.91, cy + 0.43, 2.0)]
    # seams and corners, several headings
    k = 0
    for x in (0.0, 1e-9, W - 1e-9, float(W)):
        for y in (0.0, 1e-9, H - 1e-9, float(H)):
            sites.append((x, y, SEAM_THETAS[k % len(SEAM_THETAS)]))
            k += 1
    sites += [(0.0, gy, 1000.123), (float(W), gy + 1.0, DOWN), (gx + 1.0, float(H), 0.3), (gx - 1.0, 1e-9, -999.77)]
    # next to the rocks of _rocks (harmless without rocks)
    c0x, c0y = W // 2, H // 4
    sites.append((c0x + 0.37, c0y + r + 1.37, DOWN))                  # window holds samples exactly at rock 0's radius
    mx, my = W // 4 + 0.43, 3 * H // 5 + 0.12
    sites.append((mx, my, DOWN))                                       # window that three rocks reach
    sites.append((W - 1e-9, 3 * H // 4 + 0.43, DOWN))                  # window wraps onto the rock at x = 1
    sites.append((3 * W // 4 + 0.43, 1e-9, DOWN))                      # ... and onto the rock at y = H - 1
    return sites


def _rocks(cfg, ants_xy, rng):
    """(centres, radii) of cfg's rocks: the designed ones first, the rest a lattice of small rocks clear of the ants."""
    W, H, R = cfg["w"], cfg["h"], cfg["n_rocks"]
    if R == 0:
        return np.zeros((0, 2)), np.zeros(0)
    assert R >= 6
    mx, my = W // 4 + 0.43, 3 * H // 5 + 0.12
    c = np.zeros((R, 2))
    rad = np.zeros(R)
    c[0], rad[0] = (W // 2, H // 4), 2.0                               # integer centre and radius
    c[2], rad[2] = (1.0, 3 * H // 4), 2.5                              # one cell from the x seam
    c[3], rad[3] = (3 * W // 4, H - 1.0), 2.5                          # one cell from the y seam
    multi = (1, R // 2 + 1, R - 1)                                     # (bit 63 of the masks with 64 rocks)
    for i, (dx, dy) in zip(multi, ((-2.5, 0.3), (2.6, -0.2), (0.1, 2.7))):
        c[i], rad[i] = (mx + dx, my + dy), 1.2
    free = [i for i in range(R) if rad[i] == 0.0]
    lattice = [(x + 0.25, y + 0.75) for x in range(2, W - 1, 3) for y in range(2, H - 1, 3)]
    rng.shuffle(lattice)
    for p in lattice:
        if not free:
            break
        if np.all(np.hypot(ants_xy[:, 0] - p[0], ants_xy[:, 1] - p[1]) > 1.5):
            c[free[0]], rad[free[0]] = p, 0.7
            free.pop(0)
    assert not free, "no room for %d rocks" % len(free)
    d = np.hypot(ants_xy[:, None, 0] - c[None, :, 0], ants_xy[:, None, 1] - c[None, :, 1])
    assert np.all(d > rad[None, :] + 0.05), "an ant inside a rock would push it"
    return c, rad


def edge_world(cfg, seed):
    """One env's complete state (OracleEnv / stack_init schema).  Env `seed` takes sites seed*N .. seed*N + N - 1 of
    the site list (cyclically); the map contents are drawn from `seed` around them."""
    rng = np.random.RandomState(1000 + seed)
    W, H, N = cfg["w"], cfg["h"], cfg["n_ants"]
    sites = _sites(cfg)
    pick = [sites[(seed * N + k) % len(sites)] for k in range(N)]
    x = np.array([p[0] for p in pick])
    y = np.array([p[1] for p in pick])
    theta = np.array([p[2] for p in pick])
    ax, ay, ar = seed % 2, 2, 3                                        # the disc crosses both seams
    xs, ys = np.arange(W)[:, None], np.arange(H)[None, :]
    hill = ((ax - xs) ** 2 + (ay - ys) ** 2) ** 0.5 <= ar
    ant_cells = np.zeros((W, H), bool)
    ant_cells[x.astype(int) % W, y.astype(int) % H] = True
    walls = (rng.random_sample((W, H)) < 0.12) & ~hill & ~ant_cells
    food = np.where(rng.random_sample((W, H)) < 0.4, rng.choice(FOOD_CLASSES[1:], (W, H)), 0.0)
    food[walls | hill] = 0.0
    phero = np.where(rng.random_sample((2, W, H)) < 0.25, rng.choice(PHERO_VALUES, (2, W, H)), 0.0)
    phero[:, walls] = 0.0
    explored = (rng.random_sample((W, H)) < 0.2).astype(np.uint8)
    holding = np.where(rng.random_sample(N) < 0.3, 2.5, 0.0)
    world = {"x": x, "y": y, "theta": theta, "walls": walls.astype(np.uint8), "food": food, "phero": phero,
             "explored": explored, "anthill_xyr": np.array([ax, ay, ar], np.int32), "holding": holding,
             "mandibles": (holding > 0).astype(np.uint8) * rng.randint(0, 2, N).astype(np.uint8),
             "seed": rng.random_sample(N), "activation": rng.choice([0.0, 10.0], (N, 2)), "act_bool": False}
    if cfg["n_rocks"]:
        c, rad = _rocks(cfg, np.stack([x, y], 1), rng)
        world.update(rock_centers=c, rock_radii=rad, rock_weights=rng.random_sample(cfg["n_rocks"]) * 50 + 50)
    return world


def edge_worlds(cfg, n_envs, seed0=0):
    return [edge_world(cfg, seed0 + e) for e in range(n_envs)]


# ------------------------------------------------------------------------------------------------ coverage (CPU)
def coverage(cfg, worlds):
    """Counts of every edge class over the first observation of `worlds`, from the oracle's own arithmetic."""
    W, H, r = cfg["w"], cfg["h"], cfg["radius"]
    cnt = {k: 0 for k in ("tie_x_pos", "tie_x_neg", "tie_x_centre", "tie_x_off_centre", "tie_y_pos", "tie_y_neg",
                          "near_tie", "wrap_x_low", "wrap_x_high", "wrap_y_low", "wrap_y_high", "corner", "x_is_W",
                          "y_is_H", "wall", "hill_across_seam", "ants_shared_cell", "plain_phero_below_cut",
                          "phero_max_val", "plain_phero_other", "pre_explored", "shared_unexplored",
                          "duplicate_cell", "rock_at_radius", "multi_rock", "far_rock_bit", "seam_rock")}
    cnt.update({"food_%g" % v: 0 for v in FOOD_CLASSES})
    vis = np.ones((2 * r + 1,) * 2, bool) if cfg["mask"] is None else np.asarray(cfg["mask"], bool)
    for w in worlds:
        o = OracleEnv(cfg, w)
        s = o.s
        pts = o.sample_points()
        cells = o.sample_cells()
        raw = np.round(pts).astype(int)
        frac = pts - np.floor(pts)
        tie = frac == 0.5
        cnt["near_tie"] += int(((np.abs(frac - 0.5) < NEAR_TIE) & ~tie).sum())
        for a, n in ((0, "x"), (1, "y")):
            cnt["tie_%s_pos" % n] += int((tie[..., a] & (pts[..., a] > 0)).sum())
            cnt["tie_%s_neg" % n] += int((tie[..., a] & (pts[..., a] < 0)).sum())
        cnt["tie_x_centre"] += int(tie[:, :, r, 0].sum())
        cnt["tie_x_off_centre"] += int(tie[..., 0].sum() - tie[:, :, r, 0].sum())
        cnt["wrap_x_low"] += int((raw[..., 0] < 0).sum())
        cnt["wrap_x_high"] += int((raw[..., 0] >= W).sum())
        cnt["wrap_y_low"] += int((raw[..., 1] < 0).sum())
        cnt["wrap_y_high"] += int((raw[..., 1] >= H).sum())
        wx = (raw[..., 0] < 0) | (raw[..., 0] >= W)
        wy = (raw[..., 1] < 0) | (raw[..., 1] >= H)
        cnt["corner"] += int((wx & wy).sum())
        cnt["x_is_W"] += int((s["x"] == W).sum())
        cnt["y_is_H"] += int((s["y"] == H).sum())
        cx, cy = cells[..., 0], cells[..., 1]
        seen = np.broadcast_to(vis, cx.shape)
        cnt["wall"] += int((s["walls"][cx, cy].astype(bool) & seen).sum())
        ax, ay, ar = s["anthill_xyr"]
        if ax - ar < 0 and ay - ar < 0:
            cnt["hill_across_seam"] += int((o.area[cx, cy] & seen).sum())
        amap = np.zeros((W, H), int)
        np.add.at(amap, (s["x"].astype(int) % W, s["y"].astype(int) % H), 1)
        cnt["ants_shared_cell"] += int(((amap[cx, cy] >= 2) & seen).sum())
        for v in FOOD_CLASSES:
            cnt["food_%g" % v] += int(((s["food"][cx, cy] == v) & seen).sum())
        ph = s["phero"][:, cx, cy]
        cnt["plain_phero_below_cut"] += int(((ph > 0) & (ph < 0.01) & seen).sum())
        cnt["phero_max_val"] += int(((ph == cfg["phero_max_val"]) & seen).sum())
        cnt["plain_phero_other"] += int(((ph >= 0.01) & (ph < cfg["phero_max_val"]) & seen).sum())
        unexplored = s["explored"][cx, cy] == 0
        cnt["pre_explored"] += int((~unexplored).sum())
        flat = cx * H + cy
        seen_by = {}
        for a in range(flat.shape[0]):
            for c in set(flat[a][unexplored[a]].tolist()):
                seen_by[c] = seen_by.get(c, 0) + 1
            cnt["duplicate_cell"] += int(flat[a].size - np.unique(flat[a]).size)
        cnt["shared_unexplored"] += sum(1 for v in seen_by.values() if v >= 2)
        if cfg["n_rocks"]:
            c, rad = s["rock_centers"], s["rock_radii"]
            d = np.sum((cells[:, :, :, None, :] - c[None, None, None]) ** 2, axis=4) ** 0.5    # RL_api.py:132-135
            cnt["rock_at_radius"] += int((d == rad).sum())
            hit = d < rad
            cnt["multi_rock"] += int((hit.any(axis=(1, 2)).sum(axis=1) >= 3).sum())
            cnt["far_rock_bit"] += int(hit[..., 32:].sum())
            near_seam = (c[:, 0] < 2) | (c[:, 0] > W - 2) | (c[:, 1] < 2) | (c[:, 1] > H - 2)
            cnt["seam_rock"] += int(hit[..., near_seam].sum())
    return cnt


def required_classes(cfg):
    keys = ["tie_x_pos", "tie_x_neg", "tie_x_centre", "tie_x_off_centre", "tie_y_pos", "tie_y_neg", "wrap_x_low",
            "wrap_x_high", "wrap_y_low", "wrap_y_high", "corner", "x_is_W", "y_is_H", "wall", "hill_across_seam",
            "ants_shared_cell", "plain_phero_below_cut", "phero_max_val", "plain_phero_other", "pre_explored",
            "shared_unexplored"] + ["food_%g" % v for v in FOOD_CLASSES]
    if cfg["n_rocks"]:
        keys += ["rock_at_radius", "multi_rock", "seam_rock"] + (["far_rock_bit"] if cfg["n_rocks"] > 32 else [])
    if min(cfg["w"], cfg["h"]) < 2 * cfg["radius"] + 1:
        keys.append("duplicate_cell")
    return keys


# (E, N): N odd, E * N mod 4 in {1, 3, 2}: 4-ant chunks and 32-ant warps span envs
SHAPES = ((5, 33), (37, 3), (6, 11))
RECORDS = ("f64", "compact", "compact8")
ROW_CASES = [(rec, C, S) for S in (7, 5) for C in (6, 7) for rec in RECORDS]


def row_case(rec, C, S):
    """cfg, E of a row-kernel instance: 64 rocks with the 7x7 window, 6 with the 5x5 one; the explore reward with 5x5"""
    k = ROW_CASES.index((rec, C, S))
    E, N = SHAPES[k % len(SHAPES)]
    cfg = edge_cfg(N, radius=S // 2, n_rocks=0 if C == 6 else (64 if S == 7 else 6),
                   reward_kind="all" if S == 7 else "explore")
    return cfg, E


GENERIC_EXTRA = {
    "radius1": dict(radius=1, mask=None),
    "radius4": dict(radius=4, n_rocks=6),
    "no_mask": dict(radius=3, mask=None, reward_kind="explore"),
    "permuted": dict(radius=3, n_rocks=6, channels=["food", "rocks", "phero1", "walls", "ants", "anthill", "phero0"]),
}


def threshold_sizes():
    """(W, H, slow): a map of floor(reach) and one of floor(reach) + 1 cells on each axis, default channels, 7x7."""
    reach = reach_of(edge_cfg(9))
    lo = int(np.floor(reach))
    return [(lo, 20, True), (20, lo, True), (lo + 1, 20, False), (20, lo + 1, False)]


def all_batches():
    out = [("row_%s_C%d_S%d" % (rec, C, S),) + row_case(rec, C, S) for rec, C, S in ROW_CASES]
    out += [("generic_" + k, edge_cfg(11, **kw), 6) for k, kw in GENERIC_EXTRA.items()]
    out += [("wrap_%dx%d" % (w, h), edge_cfg(9, w=w, h=h), 7) for w, h, _ in threshold_sizes()]
    return out


@pytest.mark.parametrize("name,cfg,E", all_batches(), ids=[b[0] for b in all_batches()])
def test_edge_worlds_cover_every_class(name, cfg, E):
    cnt = coverage(cfg, edge_worlds(cfg, E))
    missing = [k for k in required_classes(cfg) if cnt[k] == 0]
    assert not missing, "%s: no %s; counts %r" % (name, missing, cnt)
    assert cnt["near_tie"] == 0, "%s: %d samples within %g of a half; counts %r" % (name, cnt["near_tie"], NEAR_TIE, cnt)


def test_threshold_sizes_straddle_the_slow_wrap():
    reach = reach_of(edge_cfg(9))
    for w, h, slow in threshold_sizes():
        assert (w <= reach or h <= reach) == slow, (w, h, reach)


def test_group_ranges_are_misaligned():
    starts = {groups: group_starts(ROLL_E, ROLL_N, groups) for groups in (3, 4)}
    for groups, s in starts.items():
        ants = [e * ROLL_N for e in s]
        assert any(a % 2 == 1 for a in ants) and any(a % 4 == 2 for a in ants), (groups, ants)


# ------------------------------------------------------------------------------------------------ GPU
def oracle_step(o, ph):
    """OracleEnv.step with None rotations, cell W (H) read as cell 0: np.mod can return W itself (Q14), where the
    reference would raise IndexError; the CUDA path maps it to cell 0 (DESIGN.md section 7)."""
    s, W, H = o.s, o.cfg["w"], o.cfg["h"]
    prev = s["prev_x"].copy(), s["prev_y"].copy()
    for k, n in (("x", W), ("y", H), ("prev_x", W), ("prev_y", H)):
        s[k] = np.where(s[k] == n, 0.0, s[k])
    out = o.step(None, ph)
    s["prev_x"], s["prev_y"] = prev
    return out


def check_outputs(cfg, gpu, refs, what):
    """gpu: (obs, agent_state, reward[, state]) tensors; refs: per env (perception, agent_state, reward[, state])."""
    g = [t.cpu().numpy() for t in gpu]
    obs, ref = g[0], np.stack([r[0] for r in refs])
    ph = np.array([c.startswith("phero") for c in cfg["channels"]])
    a, b = obs[..., ~ph], ref[..., ~ph].astype(np.float32)
    bad = np.argwhere(a != b)
    assert bad.size == 0, "%s: %d non-pheromone observation entries differ, first (env, ant, i, j, ch) %r: %r vs %r" % (
        what, len(bad), tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])
    np.testing.assert_allclose(obs[..., ph], ref[..., ph], rtol=1e-5, atol=0, err_msg=what + ": pheromone channels")
    assert np.array_equal(g[1], np.stack([r[1] for r in refs]).astype(np.float32)), what + ": agent_state"
    rew = np.stack([r[2] for r in refs])
    if cfg["reward_kind"] == "explore":
        assert np.array_equal(g[2] * 10, rew * 10), what + ": explore reward"
    else:
        np.testing.assert_allclose(g[2], rew, rtol=1e-12, atol=0, err_msg=what + ": reward")
    if len(g) > 3:
        assert np.array_equal(g[3], np.stack([r[3] for r in refs]).astype(np.float32)), what + ": state"


def run_edges(cfg, E, record, steps=3, seed0=0):
    """observe, then `steps` x [step; update] with None rotations, random pheromone actions and taped noise; every
    output and the full exported state compared with the oracle after every call."""
    import torch
    from antsrl_b200 import BatchedAnts
    worlds = edge_worlds(cfg, E, seed0)
    oracles = [OracleEnv(cfg, w) for w in worlds]
    b = BatchedAnts(cfg, E, evap_mode="lazy", record=record)
    try:
        b.import_state(stack_init(cfg, worlds))
        obs, ast, st, rew = b.observe()
        refs = []
        for o in oracles:
            p_, a_, s_ = o.observation()
            refs.append((p_, a_, o.s["rewards"].copy(), s_))
        check_outputs(cfg, (obs, ast, rew, st), refs, "observe")
        compare_state(b.export_state(), oracles, "after observe", cfg)
        rng = np.random.RandomState(77)
        for t in range(steps):
            ph = rng.randint(0, 3, (E, cfg["n_ants"])).astype(np.int8)
            refs = [oracle_step(o, ph[e].astype(np.int64)) for e, o in enumerate(oracles)]
            obs, ast, rew, _ = b.step(None, torch.from_numpy(ph).cuda())
            check_outputs(cfg, (obs, ast, rew), [(r[0], r[1], r[2].copy()) for r in refs], "step %d" % t)
            compare_state(b.export_state(), oracles, "after step %d" % t, cfg)
            noise = rng.random_sample((E, cfg["n_ants"]))
            for e, o in enumerate(oracles):
                o.update(noise[e])
            b.update(torch.from_numpy(noise).cuda())
            compare_state(b.export_state(), oracles, "after update %d" % t, cfg)
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("rec,C,S", ROW_CASES, ids=["%s_C%d_S%d" % c for c in ROW_CASES])
def test_row_kernel_edges(rec, C, S):
    """Every instance of k_perceive_rows (record x layout x window) on the edge worlds."""
    cfg, E = row_case(rec, C, S)
    run_edges(cfg, E, rec)


@pytest.mark.gpu
@pytest.mark.parametrize("rec,C,S", ROW_CASES, ids=["%s_C%d_S%d" % c for c in ROW_CASES])
def test_generic_kernel_edges(rec, C, S, monkeypatch):
    """The same worlds through the generic k_perceive (ANTS_PERCEIVE_GENERIC)."""
    monkeypatch.setenv("ANTS_PERCEIVE_GENERIC", "1")
    cfg, E = row_case(rec, C, S)
    run_edges(cfg, E, rec, seed0=3)


@pytest.mark.gpu
@pytest.mark.parametrize("rec", RECORDS)
@pytest.mark.parametrize("name", sorted(GENERIC_EXTRA))
def test_generic_kernel_only_configs(name, rec):
    """Windows, masks and channel lists the row kernel never serves: radius 1 and 4, no mask, a permuted list."""
    run_edges(edge_cfg(11, **GENERIC_EXTRA[name]), 6, rec)


@pytest.mark.gpu
@pytest.mark.parametrize("rec", ("compact8", "f64"))
@pytest.mark.parametrize("w,h,slow", threshold_sizes(), ids=["%dx%d" % s[:2] for s in threshold_sizes()])
def test_maps_at_the_single_wrap_threshold(w, h, slow, rec):
    """Maps of floor(reach) cells on an axis take the generic kernel's slow wrap (a window may hold a cell twice); one
    cell more and the row kernel's single conditional wrap serves them."""
    cfg = edge_cfg(9, w=w, h=h)
    assert (w <= reach_of(cfg) or h <= reach_of(cfg)) == slow
    run_edges(cfg, 7, rec)


# grouped rollouts: N = 11 puts 256 // 11 = 23 envs in a block of the block-per-env kernel; groups start at multiples
# of 23 envs, i.e. at ants 253 (odd: C = 6 misaligned) and 506 (= 2 mod 4: C = 7 misaligned)
ROLL_E, ROLL_N = 80, 11


def group_starts(E, N, want):
    """First env of every group, as ensure_groups (ants_abi.cu) cuts a batch of N <= 256 ants per env."""
    g = max(1, min(32, 256 // N))                 # envs per block of the block-per-env kernel
    blocks = -(-E // g)
    G = min(want, blocks)
    return [(blocks * k // G) * g for k in range(G)]


@pytest.mark.gpu
@pytest.mark.parametrize("groups", (3, 4))
@pytest.mark.parametrize("C", (6, 7))
def test_grouped_rollout_ranges(C, groups, monkeypatch):
    """ants_rollout as `groups` groups on streams of their own: the perception range of a group starts at env0 * N, so
    the chunks of a group start misaligned for the bulk store and take the plain-store fallback.  The last step and
    the state must equal the oracle (Philox noise) and the same steps issued through step / update, bit for bit."""
    import torch
    from antsrl_b200 import BatchedAnts
    monkeypatch.setenv("ANTS_ROLLOUT_GROUPS", str(groups))
    starts = [e * ROLL_N for e in group_starts(ROLL_E, ROLL_N, groups)]
    assert any(a % 2 == 1 for a in starts) and any(a % 4 == 2 for a in starts), starts
    T, seed = 5, 41
    cfg = edge_cfg(ROLL_N, n_rocks=0 if C == 6 else 6)
    worlds = edge_worlds(cfg, ROLL_E)
    ph = np.random.RandomState(5).randint(0, 3, (T, ROLL_E, ROLL_N)).astype(np.int8)
    ph_d = torch.from_numpy(ph).cuda().contiguous()
    outs = []
    for mode in ("rollout", "loop"):
        b = BatchedAnts(cfg, ROLL_E, evap_mode="lazy", record="compact8", rng_seed=seed)
        b.import_state(stack_init(cfg, worlds))
        b.observe()
        if mode == "rollout":
            obs, ast, rew = b.rollout(None, ph_d)
        else:
            for t in range(T):
                obs, ast, rew, _ = b.step(None, ph_d[t])
                b.update(None)
        outs.append(([v.cpu().numpy().copy() for v in (obs, ast, rew)], b.export_state()))
        b.close()
    oracles = [OracleEnv(cfg, w) for w in worlds]
    refs = []
    for e, o in enumerate(oracles):
        o.observation()
        for t in range(T):
            r = oracle_step(o, ph[t, e].astype(np.int64))
            o.update(philox_uniform(seed, e, int(o.s["timestep"]), ROLL_N))
        refs.append((r[0], r[1], r[2].copy()))
    torch_like = [torch.from_numpy(v) for v in outs[0][0]]
    check_outputs(cfg, torch_like, refs, "last step of the grouped rollout")
    compare_state(outs[0][1], oracles, "after the grouped rollout", cfg)
    for a, b_ in zip(outs[0][0], outs[1][0]):
        assert np.array_equal(a, b_), "rollout and step / update loop outputs differ"
    for k, v in outs[0][1].items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, outs[1][1][k]), "rollout and step / update loop: %s differs" % k
