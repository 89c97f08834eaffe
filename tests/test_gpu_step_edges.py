"""Step and update kernels at their edges: hand-built worlds against the oracle.

The other half of every iteration -- RLApi.step lines 178-196 and Environment.update, i.e. k_env<UPDATE, MOVE, APT> on
the block-per-env path and k_step_move, k_food_commit, k_collide, k_rocks_pushed, k_rocks_push_ants, k_deposit_commit
and k_absorb_sweep on the flat one -- holds most of the hand-made bookkeeping: the 8-byte food codec and its 0xFFFF
escape, the owner hash of the last-writer scatters (Q1), the anthill absorb queue, the rock touch chunks and rock-grid
moves, the straight-line np.mod and the five closed forms of the mandible rule.  Random scenarios reach them only by
chance.  `step_world` builds one env's complete state and scripted tapes that reach them on purpose:
  * food records crossing the escape code both ways (65534 + 1 -> 65535, 65534 + 2.5, 65540 - 5, 65539 - 5 -> 65534,
    0.5 + 2.5 -> 3, 5.25 - 5), pickups of exactly max_hold and down to 0, escaped food absorbed in the hill;
  * every mandible rule (the channel list picks it), ants that close, open and stay;
  * several ants on one prev cell, identical cells in the envs of one block, owner-hash keys that share a slot and
    probe chains that wrap past the last slot;
  * drops queued in a disc that crosses both seams, more queued cells than an env's segment holds, a new episode of a
    window of envs between a step and the update (D1), two steps whose queue outgrows the batch-wide list (D2);
  * wall hits across the seams, on consecutive updates (theta leaves [0, 2 pi), Q3), from the move's wall flag and
    from the record; headings of +-1000 kept through a None rotation and then rotated (the far branch of pymod);
  * rocks at exactly their radius and under an ant's centre, touched by ant chunks 0 and 31 and in two envs of a block,
    pushed off the map and into the next rock-grid block, the 64th rock; ants pushed across a seam onto W itself and
    into a wall (walls come before rocks: the ant deposits there, the next update zeroes it);
  * moves onto W (from -1.1e-16) and onto 0, from W, backwards, on a one-cell-wide map (the pymod fallback);
  * deposits onto boxed and plain lazy records, bool activations, activate_all_pheromones values 0.005, 254.9, 300;
    reward_state 255 -> 229.
`Q14Oracle` is the oracle with cell W (H) read as cell 0 in step and update while the coordinate itself is kept, as
the CUDA path does (the reference raises IndexError there).  The CPU test replays every batch on it and asserts that
each class occurs; the GPU tests run the same worlds through the fused kernels (every block shape), ants_rollout, the
flat kernels and the eager and diffusion fields, comparing every output and the whole state after every call, and
food / holding / anthill_food exactly wherever the oracle's value is an integer below 2**24."""
from collections import Counter

import numpy as np
import pytest
from scipy.signal import convolve2d

from oracle.antsrl_oracle import AX, OracleEnv, anthill_area, make_config, philox_uniform
from parity_util import compare_state, stack_init
from test_gpu_perception_edges import check_outputs

TWO_PI = 2 * np.pi
ESC = 65535.0                                   # the 8-byte record's food escape code (ants_kernels.cuh kFoodEsc)
W0, H0 = 40, 35
HILL = (1, 2, 4)                                # the disc crosses both seams
ALT_HILL = (20, 28, 3)                          # the disc of the replacement episode (D1)
ACTS = (0.005, 254.9, 300.0, 0.0, 10.0)         # activate_all_pheromones values
MODE_CHANNELS = {                               # mandible rule (RL_api.py:180-184, Q5): 0 none, 1 OR, 2 AND, 3, 4
    0: ["ants", "phero0", "phero1", "walls"],
    1: ["ants", "phero0", "phero1", "walls", "food"],
    2: ["ants", "phero0", "phero1", "anthill", "walls"],
    3: ["ants", "phero0", "phero1", "food", "walls", "anthill"],
    4: ["ants", "phero0", "phero1", "anthill", "walls", "food"],
}


def rule_mode(channels):
    """The closed form k_env picks: 0 none, 1 (m | f), 2 (m & !h), 3 (m | f) & !h, 4 (m & !h) | f."""
    mode, seen_or, seen_and = 0, False, False
    for c in channels:
        if c == "food":
            seen_or, mode = True, 4 if seen_and else 1
        elif c == "anthill":
            seen_and, mode = True, 3 if seen_or else 2
    return mode


def step_cfg(n_ants, mode=4, n_rocks=0, w=W0, h=H0, **kw):
    ch = list(MODE_CHANNELS[mode]) + (["rocks"] if n_rocks else [])
    kw.setdefault("fwd_delta", 0)
    return make_config(w, h, n_ants, n_phero=2, n_rocks=n_rocks, channels=ch, max_time=1000, **kw)


# ------------------------------------------------------------------------------------------------ the fused block
def block_cap(n):
    return 256 if n <= 256 else (512 if n <= 512 else 1024)


def plane_of(w, h):
    return (-(-w // 16) * 16) * (-(-h // 16) * 16)


def envs_per_block(cfg):
    n = cfg["n_ants"]
    g = max(1, min(32, block_cap(n) // n))
    while g > 1 and g * plane_of(cfg["w"], cfg["h"]) >= 0xFFFFFFF0:
        g -= 1
    return g


def cidx(cfg, x, y):
    """ants_kernels.cuh cidx: cells in 8 x 8 blocks."""
    nby = (-(-cfg["h"] // 16) * 16) // 8
    return ((((x >> 3) * nby) + (y >> 3)) << 6) | ((x & 7) << 3) | (y & 7)


def hash_slot(key, mask):
    """ants_env_fused.cuh env_hash_slot."""
    return ((np.asarray(key, np.uint64) * np.uint64(2654435761)) & np.uint64(0xFFFFFFFF)) >> np.uint64(11) & np.uint64(mask)


def hash_stats(cfg, cells_by_env):
    """(keys sharing a home slot with another key, keys whose linear probe wrapped past slot 2 CAP - 1) of the
    block's owner hash, inserting the (env in block) * plane + cell + 1 keys in ant order."""
    g, cap = envs_per_block(cfg), block_cap(cfg["n_ants"])
    mask, plane = 2 * cap - 1, plane_of(cfg["w"], cfg["h"])
    shared = wrapped = 0
    for b0 in range(0, len(cells_by_env), g):
        keys = []
        for el, cells in enumerate(cells_by_env[b0:b0 + g]):
            keys += [el * plane + int(c) + 1 for c in cells]
        keys = list(dict.fromkeys(keys))
        home = [int(v) for v in hash_slot(keys, mask)]
        cnt = Counter(home)
        shared += sum(1 for h in home if cnt[h] > 1)
        used = np.zeros(mask + 1, bool)
        for h in home:
            s = h
            while used[s]:
                s = (s + 1) & mask
            used[s] = True
            wrapped += s < h
    return shared, wrapped


def wrap_cells(cfg, el, avoid, n):
    """Up to n cells whose keys in block slot `el` fill the last slots of the hash table: enough of them that one
    probe chain wraps where the table has room for that (2 CAP slots against W H cells: else the ones nearest the end,
    and the other ants of the block close the chain)."""
    cap = block_cap(cfg["n_ants"])
    mask, plane = 2 * cap - 1, plane_of(cfg["w"], cfg["h"])
    W, H = cfg["w"], cfg["h"]
    cand = [(x, y) for x in range(W) for y in range(H) if not avoid[x, y]]
    home = hash_slot([el * plane + cidx(cfg, x, y) + 1 for x, y in cand], mask).astype(np.int64)
    for k in range(n - 1):
        pick = [c for c, h in zip(cand, home) if h >= mask - k]
        if len(pick) >= k + 2:
            return pick[:k + 2]
    return [cand[i] for i in np.argsort(-home, kind="stable")[:n]]


# ------------------------------------------------------------------------------------------------ worlds
def _seam_push_x(rc, rad):
    """Start x (theta = pi, one cell per step) of an ant that the heavy rock (rc, .) pushes to -tiny: np.mod puts it on
    W itself.  The oracle's arithmetic of circle_obstacles.py:32-58 for one ant and one rock of weight 1e9."""
    def final(p):
        x0 = p + np.cos(np.pi) * 1.0
        v = rc - x0
        d = (v * v) ** 0.5
        c = rc - v * (1 - rad / (d + 0.001)) / 1e9
        v = c - x0
        d = (v * v) ** 0.5
        return x0 + v * (1 - rad / (d + 0.001))
    lo, hi = 1.0 + rc - rad + 1e-3, 1.0 + rc - 1e-3
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        if final(mid) < 0:
            lo = mid
        else:
            hi = mid
    p = lo
    for _ in range(1 << 12):
        f = final(p)
        if f < 0 and np.mod(f, float(W0)) == W0:
            return p
        p = np.nextafter(p, np.inf) if f < 0 else np.nextafter(p, -np.inf)
    raise AssertionError("no start that lands on W")


SEAM_ROCK = (0.9, 12.05)


def _design(cfg, hill):
    """The designed ants (x, y, theta, prev_x, prev_y, holding, mandibles, reward_state), food, walls and rocks.  The
    first COMMON ants are the same in every env (identical cells in the envs of a block)."""
    W, H = cfg["w"], cfg["h"]
    ants, food, walls, rocks = [], {}, set(), []

    def ant(x, y, th=0.3, px=None, py=None, hold=0.0, mand=0, rs=0):
        ants.append((x, y, th, x if px is None else px, y if py is None else py, hold, mand, rs))

    in_hill = [(2.37, 3.43), (1.37, 1.43), (3.43, 4.37), (4.37, 2.43), (0.37, 5.43), (2.63, 2.61)]
    # common: a rock at exactly its radius after the move, drops queued inside the seam-crossing disc, a pickup
    ant(21.0, 10.0, 0.0)                                            # -> (22, 10): |rock 63 - ant| == 2 == radius
    ant(in_hill[3][0], in_hill[3][1], 1.1, 2.5, 1.5, hold=2.5, mand=1)     # drop 2.5 onto (2, 1): escaped, queued
    ant(in_hill[4][0], in_hill[4][1], 1.9, 0.5, 4.5, hold=4.0, mand=1)     # drop 4 onto (0, 4): queued
    ant(8.37, 16.43, 2.2)                                           # pickup 5 from 65540 -> 65535
    food[(8, 16)] = 65540.0
    # the food codec on prev cells of row 16 (pickups stand there, drops stand in the hill)
    for k, (f, hold, mand, spot) in enumerate(((65534.0, 1.0, 1, 0), (65534.0, 2.5, 1, 1), (65539.0, 0.0, 0, None),
                                               (0.5, 2.5, 1, 2), (5.25, 0.0, 0, None), (7.0, 0.0, 0, None),
                                               (3.0, 0.0, 0, None))):
        cx = 10 + 2 * k
        food[(cx, 16)] = f
        x, y = (cx + 0.37, 16.43) if spot is None else in_hill[spot]
        ant(x, y, 0.9 + 0.4 * k, cx + 0.37, 16.43, hold=hold, mand=mand)
    # several ants on one prev cell: one drops (standing in the hill), one picks up, one stays
    food[(14, 12)] = 9.0
    ant(in_hill[5][0], in_hill[5][1], 2.7, 14.37, 12.43, hold=2.0, mand=1)
    ant(14.37, 12.43, 0.7)
    ant(14.63, 12.77, 4.0, hold=1.0, mand=1)
    # walled pockets: every move leaves into a wall, across the x seam, across the y seam, and theta past 2 pi
    for (cx, cy), th in (((0, 20), np.pi + 0.1), ((20, 0), -np.pi / 2 - 0.1), ((30, 20), 6.1)):
        for dx in (-1, 0, 1):
            for dy in (-1, 0, 1):
                if dx or dy:
                    walls.add(((cx + dx) % W, (cy + dy) % H))
        ant(cx + 0.5, cy + 0.5, th)
    ant(12.37, 26.43, 1000.1)                                       # headings far outside [0, 2 pi)
    ant(16.37, 26.43, -999.8)
    walls.add((10, 30))
    ant(10.5, 30.5, 1.3, 9.5, 30.5)                                 # imported inside a wall (record read)
    # moves onto 0 from W - 1, onto W from below 0, from W and H themselves, backwards
    ant(39.0, 22.43, 0.0)
    ant(1.0 - 2.0 ** -53, 24.43, np.pi)
    ant(40.0, 28.43, 0.0)
    ant(33.37, 35.0, -np.pi / 2)
    ant(8.37, 22.43, 0.3, hold=25.0, mand=1, rs=255)
    # rocks: at the centre, off the map (light), into the next grid block, pushed onto W, pushed into a wall
    ant(24.0, 14.0, 0.0)
    ant(37.95, 25.05, 0.0)
    ant(14.05, 30.0, 0.0)
    ant(_seam_push_x(*SEAM_ROCK[:1], 1.0), SEAM_ROCK[1], np.pi)
    ant(31.05, 5.05, np.pi, rs=255)
    walls.add((29, 5))
    ant(22.0, 10.0, np.pi)                                          # (ant N - 1 for N >= 993: chunk 31 on rock 63)
    rocks = [((20.0, 10.0), 2.0, 60.0), ((25.0, 14.0), 1.5, 70.0), ((39.5, 25.0), 1.0, 0.01),
             ((15.4, 30.0), 0.4, 0.05), (SEAM_ROCK, 1.0, 1e9), ((30.75, 5.05), 1.0, 1e9)]
    # food in the disc before the first sweep (Q10)
    food[(3, 3)] = 2.0
    food[(0, 0)] = 65536.5
    return ants, food, walls, rocks


COMMON = 4


def step_world(cfg, seed, hill=HILL, old_hill=None):
    """One env's complete state.  Env `seed` takes the COMMON ants, then the rest of the designed ants cyclically from
    seed * (N - COMMON); beyond the design (N > len) random ants fill up.  The owner-hash ants (holding 20: speed 0,
    closed outside the hill, so they never move) sit on cells whose keys fill the last slots of the table for the env's
    slot in its block.  `old_hill`: food 3 on every free cell of that disc (the replacement episode of D1)."""
    rng = np.random.RandomState(500 + seed)
    W, H, N, R = cfg["w"], cfg["h"], cfg["n_ants"], cfg["n_rocks"]
    ants, food_d, walls_d, rocks_d = _design(cfg, hill)
    tiny = W < 8 or H < 8
    ax, ay, ar = hill
    xs, ys = np.arange(W)[:, AX], np.arange(H)[AX, :]
    area = ((ax - xs) ** 2 + (ay - ys) ** 2) ** 0.5 <= ar
    reserved = area.copy()
    if tiny:
        ants = []
        food_d, walls_d, rocks_d = {}, set(), []
    n_hash = 0 if tiny else (4 if N <= 256 else 8)
    n_design = N - n_hash
    pick = list(range(min(COMMON, len(ants), n_design)))
    rest = list(range(COMMON, len(ants)))
    if n_design > len(pick) and rest:
        if n_design >= len(ants):
            pick += rest
        else:
            off = seed * (n_design - len(pick))
            pick += [rest[(off + k) % len(rest)] for k in range(n_design - len(pick))]
    chosen = [ants[k] for k in pick]
    for a in ants:
        for px, py in ((a[0], a[1]), (a[3], a[4])):
            cx, cy = int(px) % W, int(py) % H
            reserved[max(cx - 1, 0):cx + 2, max(cy - 1, 0):cy + 2] = True
    for (c, rad, _) in rocks_d:
        x0, y0 = int(c[0]), int(c[1])
        reserved[max(x0 - 3, 0):x0 + 4, max(y0 - 3, 0):y0 + 4] = True
    for c in walls_d:
        reserved[c] = True
    if old_hill is not None:
        reserved |= ((old_hill[0] - xs) ** 2 + (old_hill[1] - ys) ** 2) ** 0.5 <= old_hill[2]
    # the owner-hash ants
    hash_ants = []
    if n_hash:
        el = seed % envs_per_block(cfg)
        for cx, cy in wrap_cells(cfg, el, reserved, n_hash):
            hash_ants.append((cx + 0.37, cy + 0.43, 0.5, cx + 0.37, cy + 0.43, 20.0, 1, 0))
            reserved[cx, cy] = True
        while len(hash_ants) < n_hash:
            hash_ants.append(hash_ants[-1])
    filler = []
    for k in range(N - len(chosen) - len(hash_ants)):
        while True:             # (outside the designed neighbourhoods, except on maps too small for that)
            fx, fy = rng.random_sample() * W, rng.random_sample() * H
            if tiny or not reserved[int(fx), int(fy)]:
                break
        hold = float(rng.choice([0.0, 2.5, 1.0]))
        filler.append((fx, fy, rng.random_sample() * TWO_PI, fx, fy, hold, int(hold > 0) * rng.randint(0, 2), 0))
    everyone = chosen + hash_ants + filler
    assert len(everyone) == N
    if N >= 993 and not tiny:
        everyone[-1] = ants[-1]                                     # chunk 31 with chunk 0 on rock 63
    a = np.array(everyone, dtype=float)
    x, y, th, px, py, hold, mand, rs = a.T
    n_placed = len(chosen) + len(hash_ants)
    # the map
    free = ~reserved
    walls = (rng.random_sample((W, H)) < 0.06) & free
    food = np.where((rng.random_sample((W, H)) < 0.25) & free,
                    rng.choice([1.0, 2.0, 3.0, 0.25, 65534.0, 65536.5], (W, H)), 0.0)
    for (cx, cy), v in food_d.items():
        food[cx, cy] = v
    for c in walls_d:
        walls[c] = True
    for cx, cy, _, _, _, _, _, _ in hash_ants:
        food[int(cx), int(cy)] = 2.0
    if old_hill is not None:
        od = ((old_hill[0] - xs) ** 2 + (old_hill[1] - ys) ** 2) ** 0.5 <= old_hill[2]
        food[od & ~walls] = 3.0
    food[walls] = 0.0
    phero = np.where(rng.random_sample((2, W, H)) < 0.25, rng.choice([0.005, 0.5, 3.7, 100.0, 254.9, 255.0], (2, W, H)), 0.0)
    for k in range(len(a)):                                         # saturated deposits under the ants (boxed records)
        phero[k % 2, int(x[k]) % W, int(y[k]) % H] = 255.0
    phero[:, walls] = 0.0
    act = np.array([[ACTS[k % 5], ACTS[(k + 2) % 5]] for k in range(N)])
    world = {"x": x, "y": y, "theta": th, "prev_x": px, "prev_y": py, "prev_theta": th.copy(), "holding": hold,
             "mandibles": mand.astype(np.uint8), "reward_state": rs.astype(np.uint8), "seed": rng.random_sample(N),
             "activation": act, "rw_holding_prev": np.zeros(N), "rewards": np.zeros(N),
             "walls": walls.astype(np.uint8), "food": food, "phero": phero,
             "explored": (rng.random_sample((W, H)) < 0.2).astype(np.uint8),
             "anthill_xyr": np.array(hill, np.int32), "anthill_food": np.float64(3.0 * seed)}
    if R:
        c = np.zeros((R, 2))
        rad = np.zeros(R)
        wt = rng.random_sample(R) * 50 + 50
        slots = [R - 1] + list(range(len(rocks_d) - 1))            # rock 0 of the design is the 64th rock
        for s, (cc, rr, ww) in zip(slots, rocks_d[:R]):
            c[s], rad[s], wt[s] = cc, rr, ww
        spots = [(gx + 0.25, gy + 0.75) for gx in range(2, W - 1, 3) for gy in range(2, H - 1, 3)]
        rng.shuffle(spots)
        for s in [k for k in range(R) if rad[k] == 0.0]:
            while True:
                p = spots.pop()
                if np.all(np.hypot(x[:n_placed] - p[0], y[:n_placed] - p[1]) > 1.6) and not reserved[int(p[0]), int(p[1])]:
                    break
            c[s], rad[s] = p, 0.7
        world.update(rock_centers=c, rock_radii=rad, rock_weights=wt)
    return world


def overflow_world(cfg, seed):
    """D2: rule mode 3, a radius-10 disc whose cells hold food 9, N ants on distinct cells of its rim facing outward
    with closed mandibles and 2 units each.  Step 1: all of them stand in the hill and drop (queued); step 2, without
    an update: they stand outside and pick up from the unchanged prev cell (queued again)."""
    W, H, N = cfg["w"], cfg["h"], cfg["n_ants"]
    ax, ay, ar = 20, 17, 10
    xs, ys = np.arange(W)[:, AX], np.arange(H)[AX, :]
    area = ((ax - xs) ** 2 + (ay - ys) ** 2) ** 0.5 <= ar
    rim = []
    for cx in range(W):
        for cy in range(H):
            if not area[cx, cy]:
                continue
            px, py = cx + 0.5, cy + 0.5
            th = np.arctan2(py - ay, px - ax)
            nx, ny = px + np.cos(th), py + np.sin(th)
            if not area[int(nx) % W, int(ny) % H] and min(abs(nx - round(nx)), abs(ny - round(ny))) > 1e-6:
                rim.append((np.arctan2(py - ay, px - ax), px, py, th))
    rim.sort()
    assert len(rim) >= N, "%d rim cells for %d ants" % (len(rim), N)
    sel = [rim[k * len(rim) // N] for k in range(N)]
    x = np.array([s[1] for s in sel])
    y = np.array([s[2] for s in sel])
    th = np.array([s[3] for s in sel])
    return {"x": x, "y": y, "theta": th, "holding": np.full(N, 2.0), "mandibles": np.ones(N, np.uint8),
            "seed": np.linspace(0, 1, N), "activation": np.zeros((N, 2)), "rw_holding_prev": np.zeros(N),
            "rewards": np.zeros(N), "reward_state": np.zeros(N, np.uint8),
            "walls": np.zeros((W, H), np.uint8), "food": np.where(area, 9.0, 0.0), "phero": np.zeros((2, W, H)),
            "explored": np.zeros((W, H), np.uint8), "anthill_xyr": np.array([ax, ay, ar], np.int32),
            "anthill_food": np.float64(seed)}


def tapes(cfg, worlds, T, seed=3):
    """(rot, rot_none, ph, ph_none, noise): step 0 keeps the imported headings and activations (None actions); the
    walled-pocket ants draw 0.95 (theta grows past 2 pi)."""
    rng = np.random.RandomState(seed)
    E, N = len(worlds), cfg["n_ants"]
    rot = rng.randint(-1, 2, (T, E, N)).astype(np.int8)
    ph = rng.randint(0, 3, (T, E, N)).astype(np.int8)
    noise = rng.random_sample((T, E, N))
    for e, w in enumerate(worlds):
        pocket = (w["theta"] == 6.1) | (w["theta"] == np.pi + 0.1) | (w["theta"] == -np.pi / 2 - 0.1)
        noise[:, e, pocket] = 0.95
        axis = (w["theta"] == 0.0) | (w["theta"] == np.pi)
        rot[1:, e, axis] = 1        # headings along an axis only for the designed first move (exact sample grids)
    rot_none = np.array([t % 2 == 0 for t in range(T)])
    ph_none = np.array([t == 0 for t in range(T)])
    return rot, rot_none, ph, ph_none, noise


# ------------------------------------------------------------------------------------------------ the oracle, Q14
class Q14Oracle(OracleEnv):
    """OracleEnv.step / update with the cells of x == W (y == H) read as cell 0 and the coordinate kept (Q14: np.mod can
    return W; the reference raises IndexError there, the CUDA path maps it to cell 0 and moves on from W).  The code
    follows OracleEnv line by line; `ev` counts the edge classes this file builds."""

    def __init__(self, cfg, state):
        super().__init__(cfg, state)
        self.ev = Counter()
        self.queued = 0                 # absorb entries k_food_commit would append since the last update
        self.moved = False              # a step ran since the last update (the update then uses the wall flag)
        self.hit_last = np.zeros(cfg["n_ants"], bool)
        self.mode = rule_mode(cfg["channels"])

    def cells(self, xk="x", yk="y"):
        return self.s[xk].astype(int) % self.cfg["w"], self.s[yk].astype(int) % self.cfg["h"]

    def step(self, rotation, pheromone):
        s, cfg, ev = self.s, self.cfg, self.ev
        w, h, n = cfg["w"], cfg["h"], cfg["n_ants"]
        pcx, pcy = self.cells("prev_x", "prev_y")                                  # :178
        cx, cy = self.cells()
        f = s["food"][pcx, pcy]
        m = s["mandibles"].astype(np.int64)
        for ch in cfg["channels"]:                                                # :180-184 (Q5)
            if ch == "food":
                m = np.bitwise_or(f > 0, m)
            elif ch == "anthill":
                m = np.bitwise_and(1 - self.area[cx, cy], m)
        old = s["mandibles"].astype(np.int64)
        closing = np.bitwise_and(m, 1 - old)
        opening = np.bitwise_and(1 - m, old)
        s["mandibles"] = m.astype(np.uint8)
        taken = np.minimum(cfg["max_hold"], np.maximum(0, f)) * closing
        dropped = s["holding"].copy() * opening
        before = s["food"].copy()
        s["food"][pcx, pcy] += dropped - taken                                    # last ant wins, Q1
        s["holding"] = s["holding"] + (taken - dropped)
        # -- classes
        md = "mode%d_" % self.mode
        ev[md + "close"] += int(closing.sum())
        ev[md + "open"] += int(opening.sum())
        ev[md + "stay"] += int((m == old).sum())
        delta = dropped - taken
        flat = pcx * h + pcy
        last = np.full(w * h, -1)
        last[flat] = np.arange(n)
        chg = (last[flat] == np.arange(n)) & (delta != 0)
        o, nv = before[pcx, pcy], s["food"][pcx, pcy]
        isint = lambda v: v == np.floor(v)
        ev["codec_to_esc"] += int((chg & (o < ESC) & (nv == ESC)).sum())
        ev["codec_over_esc"] += int((chg & (o < ESC) & (nv > ESC) & ~isint(nv)).sum())
        ev["codec_down_to_esc"] += int((chg & (o > ESC) & (nv == ESC)).sum())
        ev["codec_back_to_code"] += int((chg & (o > ESC) & (nv < ESC) & isint(nv)).sum())
        ev["codec_frac_to_int"] += int((chg & ~isint(o) & isint(nv) & (delta > 0)).sum())
        ev["codec_frac_left"] += int((chg & ~isint(o) & ~isint(nv) & (delta < 0)).sum())
        ev["pickup_max_hold"] += int((taken == cfg["max_hold"]).sum())
        ev["pickup_to_zero"] += int((chg & (delta < 0) & (nv == 0)).sum())
        q = chg & (nv != 0) & self.area[pcx, pcy]
        self.queued += int(q.sum())
        ev["hill_queue_drop"] += int((q & (delta > 0)).sum())
        ev["hill_queue_escaped"] += int((q & (~isint(nv) | (nv >= ESC))).sum())
        cnt = np.bincount(flat, minlength=w * h)
        shared = cnt[flat] >= 2
        ev["shared_prev_change"] += int((shared & (delta != 0)).sum())
        mixed = np.zeros(w * h, int)
        np.bitwise_or.at(mixed, flat, (taken > 0) * 1 + (dropped > 0) * 2)
        ev["shared_prev_mixed"] += int((mixed == 3).sum())
        # -- the move
        if pheromone is not None:                                                 # ants.py:89-96
            ph = np.asarray(pheromone)
            on = 1.0 if s["act_bool"] else 256.0
            act = np.zeros((n, 2))
            act[ph == 1, 0] = on
            act[(ph != 0) & (ph != 1), 1] = on
            s["activation"] = act
        if rotation is not None:                                                  # ants.py:62-67
            t = s["theta"] + np.asarray(rotation) * cfg["max_rot_speed"]
            ev["theta_far_rotated"] += int(((t <= -TWO_PI) | (t >= 2 * TWO_PI)).sum())
            s["theta"] = np.mod(t, TWO_PI)
        else:
            ev["theta_far_kept"] += int(((s["theta"] < -TWO_PI) | (s["theta"] >= 2 * TWO_PI)).sum())
        fwd = np.ones(n) * cfg["max_speed"] * (1 - s["holding"] * cfg["carry_speed_reduction"])
        ev["backward"] += int((fwd < 0).sum())
        fwd[fwd < 0] *= cfg["backward_speed_reduction"]
        ev["move_from_W"] += int(((s["x"] == w) | (s["y"] == h)).sum())
        nx = s["x"] + np.cos(s["theta"]) * fwd
        ny = s["y"] + np.sin(s["theta"]) * fwd
        ev["move_far"] += int(((nx >= 2 * w) | (nx <= -w) | (ny >= 2 * h) | (ny <= -h)).sum())
        s["x"] = np.mod(nx, w)
        s["y"] = np.mod(ny, h)
        ev["move_to_W"] += int(((s["x"] == w) & (nx < 0)).sum() + ((s["y"] == h) & (ny < 0)).sum())
        ev["move_to_0"] += int(((s["x"] == 0) & (nx == w)).sum() + ((s["y"] == 0) & (ny == h)).sum())
        self.moved = True
        perception, agent_state, _ = self.observation()                           # :198 (Q2)
        done = cfg["max_time"] == int(s["timestep"])
        reward = s["rewards"]
        add = ((reward - cfg["reward_threshold"]) > 0) * 255
        s["reward_state"] = np.minimum(s["reward_state"].astype(np.int64) + add, 255).astype(np.uint8)
        return perception, agent_state, reward, bool(done)

    def update(self, noise=None):
        s, cfg, ev = self.s, self.cfg, self.ev
        w, h, n = cfg["w"], cfg["h"], cfg["n_ants"]
        s["timestep"] = int(s["timestep"]) + 1
        walls = s["walls"].astype(bool)
        cx, cy = self.cells()
        hit = walls[cx, cy]                                                       # walls.py:22-30
        ev["wall_hit_" + ("flag" if self.moved else "record")] += int(hit.sum())
        ev["wall_hit_seam"] += int((hit & ((np.abs(s["x"] - s["prev_x"]) > w / 2) |
                                           (np.abs(s["y"] - s["prev_y"]) > h / 2))).sum())
        ev["wall_hit_again"] += int((hit & self.hit_last).sum())
        self.hit_last = hit
        if hit.any():
            s["x"] = np.where(hit, s["prev_x"], s["x"])
            s["y"] = np.where(hit, s["prev_y"], s["y"])
            th = s["theta"].copy()
            th[hit] += np.asarray(noise, dtype=float)[hit] - 0.5                  # Q3
            s["theta"] = th
            ev["theta_outside"] += int((hit & ((th < 0) | (th >= TWO_PI))).sum())
        ev["deposit_on_wall_zeroed"] += int((s["phero"][:, walls] > 0).sum())
        for p in range(cfg["n_phero"]):
            s["phero"][p][walls] = 0
        if cfg["n_rocks"] > 0:                                                    # circle_obstacles.py:32-58
            c, rad, wt = s["rock_centers"], s["rock_radii"], s["rock_weights"]
            xy = np.stack([s["x"], s["y"]], axis=1)
            v = c[AX, :, :] - xy[:, AX, :]
            d = np.sum(v ** 2, axis=2) ** 0.5
            ev["rock_at_radius"] += int((d == rad[AX, :]).sum())
            ev["ant_at_rock_centre"] += int((d == 0).sum())
            touch = ~(d > rad[AX, :])
            gc = ((n + 31) // 32 + 31) // 32 * 32
            ev["rock_chunks_0_31"] += int((touch[:gc].any(0) & touch[31 * gc:].any(0)).sum()) if n > 31 * gc else 0
            ev["rock_64_touched"] += int(touch[:, 63].any()) if cfg["n_rocks"] >= 64 else 0
            push = v * (1 - rad[AX, :] / (d + 0.001))[:, :, AX]
            push[d > rad[AX, :], :] = 0
            c0 = c
            c = c - np.sum(push, axis=0) / wt[:, AX]
            s["rock_centers"] = c
            moved = np.any(c != c0, axis=1)
            off = (c[:, 0] < 0) | (c[:, 0] >= w) | (c[:, 1] < 0) | (c[:, 1] >= h)
            ev["rock_off_map"] += int((moved & off).sum())
            ev["rock_grid_block"] += int((moved & np.any(np.floor(c / 16) != np.floor(c0 / 16), axis=1)).sum())
            v = c[AX, :, :] - xy[:, AX, :]
            d = np.sum(v ** 2, axis=2) ** 0.5
            push = v * (1 - rad[AX, :] / (d + 0.001))[:, :, AX]
            push[d > rad[AX, :], :] = 0
            pushed = np.any(d <= rad[AX, :], axis=1)
            xy = xy + np.sum(push, axis=1)
            s["x"] = np.mod(xy[:, 0], w)
            s["y"] = np.mod(xy[:, 1], h)
            ev["pushed_onto_W"] += int((pushed & ((s["x"] == w) | (s["y"] == h))).sum())
            ncx, ncy = self.cells()
            ev["pushed_into_wall"] += int((pushed & walls[ncx, ncy] & ~walls[cx, cy]).sum())
        for p in range(cfg["n_phero"]):                                           # pheromone.py:43-45
            ph = convolve2d(s["phero"][p], self.filter, 'same', 'fill', 0)
            ph[ph < 0.01] = 0
            s["phero"][p] = ph
        s["prev_x"], s["prev_y"], s["prev_theta"] = s["x"].copy(), s["y"].copy(), s["theta"].copy()
        cx, cy = self.cells()
        last = np.full(w * h, -1)
        last[cx * h + cy] = np.arange(n)
        own = last[cx * h + cy] == np.arange(n)
        for p in range(cfg["n_phero"]):                                           # ants.py:123-130, pheromone.py:36-41
            a = s["activation"][:, p]
            dep = own & (a > 0)
            before = s["phero"][p][cx, cy]
            ev["deposit_on_wall"] += int((dep & walls[cx, cy]).sum())
            ev["deposit_on_saturated"] += int((dep & (before >= cfg["phero_max_val"] * 0.99)).sum())
            ev["deposit_clamped"] += int((dep & (before + a >= cfg["phero_max_val"])).sum())
            ev["deposit_1"] += int((dep & (a == 1.0)).sum())
            for v in ACTS[:3]:
                ev["deposit_%g" % v] += int((dep & (a == v)).sum())
            s["phero"][p][cx, cy] += a
            s["phero"][p] = np.minimum(s["phero"][p], cfg["phero_max_val"])
        ev["reward_state_255"] += int((s["reward_state"] == 255).sum())
        s["reward_state"] = (s["reward_state"] * 0.9).astype(np.uint8)            # Q16
        gain = s["food"] * self.area                                              # anthill.py:41-46
        ev["absorb_escaped"] += int(((gain != 0) & ((gain != np.floor(gain)) | (gain >= ESC))).sum())
        ev["queue_over_N"] += int(self.queued > n)
        s["food"] -= gain
        s["anthill_food"] = np.float64(s["anthill_food"] + np.sum(gain))
        self.queued = 0
        self.moved = False


def near_ties(o):
    """Samples within 1e-12 of a half without being on it (a 1-ulp libm difference could flip them)."""
    frac = o.sample_points() - np.floor(o.sample_points())
    return int(((np.abs(frac - 0.5) < 1e-12) & (frac != 0.5)).sum())


# ------------------------------------------------------------------------------------------------ batches and replay
def activations(cfg, act):
    """What the batches pass to activate_all_pheromones: the float values of ACTS (256 deposits from then on), or
    without rocks a bool array (ants.py:83: the dtype stays bool and deposits are 1.0)."""
    return act > 0 if cfg["n_rocks"] == 0 else np.asarray(act, float)


def batch_cfg(name):
    """(cfg, E) of a named batch."""
    if name.startswith("mode"):
        return step_cfg(11, mode=int(name[4])), 50
    n = {"n11": 11, "n300": 300, "n1000": 1000, "n1030": 1030}[name]
    return step_cfg(n, n_rocks=64), {11: 50, 300: 3, 1000: 2, 1030: 2}[n]


def tiny_cfg():
    return step_cfg(5, w=1, h=3, max_speed=1.9, radius=1, mask=None)


BATCHES = ["n11", "n300", "n1000", "n1030"] + ["mode%d" % m for m in range(5)]


def replay(cfg, worlds, T=4):
    """observe; activate_all_pheromones; T x [step; update] on Q14Oracle: the events of all envs, the queue entries
    between two updates summed over the envs, near ties."""
    oracles = [Q14Oracle(cfg, w) for w in worlds]
    rot, rot_none, ph, ph_none, noise = tapes(cfg, worlds, T)
    ties = 0
    queue_total = 0
    for o in oracles:
        o.observation()
        ties += near_ties(o)
    for o in oracles:
        o.activate_all_pheromones(activations(cfg, o.s["activation"]))
    for t in range(T):
        for e, o in enumerate(oracles):
            o.step(None if rot_none[t] else rot[t, e].astype(np.int64), None if ph_none[t] else ph[t, e].astype(np.int64))
            ties += near_ties(o)
        queue_total = max(queue_total, sum(o.queued for o in oracles))
        for e, o in enumerate(oracles):
            o.update(noise[t, e])
    ev = Counter()
    for o in oracles:
        ev.update(o.ev)
    return ev, queue_total, ties, oracles


REQUIRED = ["codec_down_to_esc", "codec_back_to_code", "codec_frac_left", "pickup_max_hold", "pickup_to_zero",
            "hill_queue_drop", "hill_queue_escaped", "shared_prev_change", "wall_hit_flag", "wall_hit_seam",
            "wall_hit_again", "theta_outside", "theta_far_kept", "theta_far_rotated", "move_to_W", "move_to_0",
            "move_from_W", "backward", "deposit_on_saturated", "deposit_clamped", "reward_state_255",
            "absorb_escaped"]
ROCK_REQUIRED = ["rock_at_radius", "ant_at_rock_centre", "rock_off_map", "rock_grid_block", "rock_64_touched",
                 "pushed_onto_W", "pushed_into_wall", "deposit_on_wall", "deposit_on_wall_zeroed"]


def required(cfg):
    mode = rule_mode(cfg["channels"])
    keys = [k for k in REQUIRED if not (mode in (0, 1, 2) and k in ("codec_down_to_esc", "codec_back_to_code",
                                                                    "codec_frac_left", "pickup_max_hold",
                                                                    "pickup_to_zero"))]
    if mode in (0, 1):
        keys = [k for k in keys if not k.startswith("hill_queue") and k != "absorb_escaped"]
    if mode == 0:
        keys.remove("shared_prev_change")
    keys += {0: ["mode0_stay"], 1: ["mode1_close", "mode1_stay"], 2: ["mode2_open", "mode2_stay"],
             3: ["mode3_close", "mode3_open", "mode3_stay", "codec_to_esc", "codec_over_esc", "codec_frac_to_int",
                 "shared_prev_mixed"],
             4: ["mode4_close", "mode4_open", "mode4_stay"]}[mode]
    if mode == 2:
        keys += ["codec_to_esc", "codec_over_esc", "codec_frac_to_int"]
    keys += ["deposit_1"] if cfg["n_rocks"] == 0 else ["deposit_0.005", "deposit_254.9", "deposit_300"]
    if cfg["n_rocks"]:
        keys += ROCK_REQUIRED
        if 993 <= cfg["n_ants"] <= 1024:
            keys.append("rock_chunks_0_31")
    return keys


@pytest.mark.parametrize("name", BATCHES)
def test_step_worlds_cover_every_class(name):
    cfg, E = batch_cfg(name)
    worlds = [step_world(cfg, e) for e in range(E)]
    ev, _, ties, oracles = replay(cfg, worlds)
    missing = [k for k in required(cfg) if ev[k] == 0]
    assert not missing, "%s: no %s; counts %r" % (name, missing, dict(ev))
    assert ties == 0, "%s: %d samples within 1e-12 of a half" % (name, ties)
    if cfg["n_ants"] <= 1024:       # (the keys of the update after the import: the imported cells)
        shared, wrapped = hash_stats(cfg, [[cidx(cfg, int(x) % cfg["w"], int(y) % cfg["h"])
                                            for x, y in zip(w["x"], w["y"])] for w in worlds])
        # (one env per block from N = 300 on: its W H cells hold too few keys per slot for a designed wrap)
        assert shared > 0 and (wrapped > 0 or envs_per_block(cfg) == 1), \
            "%s: owner hash: %d keys share a slot, %d wrapped" % (name, shared, wrapped)
    g = envs_per_block(cfg)
    if g > 1:       # identical cells in the envs of one block (the hash key separates them by env)
        assert np.array_equal(worlds[0]["x"][:COMMON], worlds[1]["x"][:COMMON])
        assert E % g != 0, "no partial last block"
    print(name, dict(sorted(ev.items())))


def test_tiny_map_takes_the_pymod_fallback():
    cfg = tiny_cfg()
    ev, _, ties, _ = replay(cfg, [step_world(cfg, e) for e in range(4)])
    assert ev["move_far"] > 0, dict(ev)


def test_overflow_world_queues_more_than_the_list_holds():
    """D2 on the oracle: two steps without an update queue 2 E N cells (k_food_commit's count), the list holds E N."""
    cfg = step_cfg(40, mode=3)
    E = 3
    worlds = [overflow_world(cfg, e) for e in range(E)]
    oracles = [Q14Oracle(cfg, w) for w in worlds]
    for o in oracles:
        o.observation()
        o.step(None, None)
        assert o.queued == cfg["n_ants"], o.queued
        o.step(None, None)
        assert near_ties(o) == 0
    total = sum(o.queued for o in oracles)
    print("queued between two updates: %d, list holds E * N = %d" % (total, E * cfg["n_ants"]))
    assert total == 2 * E * cfg["n_ants"] > E * cfg["n_ants"]
    for o in oracles:
        o.update(np.zeros(cfg["n_ants"]))
        assert o.ev["queue_over_N"] == 1


def test_window_episode_moves_the_disc_off_the_queued_cells():
    """D1 on the oracle: the common drops of step 0 are queued at (2, 1) and (0, 4) in every env; the replacement
    episode has food on those cells and its disc elsewhere, so the reference leaves that food where it is."""
    cfg, E = batch_cfg("n11")
    o = Q14Oracle(cfg, step_world(cfg, 1))
    o.observation()
    o.step(None, None)
    assert o.queued >= 2
    new = step_world(cfg, 101, hill=ALT_HILL, old_hill=HILL)
    assert new["food"][2, 1] == 3.0 and new["food"][0, 4] == 3.0
    n = Q14Oracle(cfg, new)
    assert not n.area[2, 1] and not n.area[0, 4]


# ------------------------------------------------------------------------------------------------ GPU
def strict_check(gpu, oracles, what, record):
    """food, holding and anthill_food exactly equal wherever the oracle's value is an integer below 2**24 (DESIGN §2:
    integer food is exact); f64 records: food exactly everywhere."""
    for k in ("food", "holding", "anthill_food"):
        ref = np.stack([np.asarray(o.s[k], float) for o in oracles])
        g = np.asarray(gpu[k], float)
        m = (ref == np.floor(ref)) & (np.abs(ref) < 2.0 ** 24)
        if k == "food" and record == "f64":
            m = np.ones_like(m)
        bad = np.argwhere(m & (g != ref))
        assert bad.size == 0, "%s: %s differs at %d entries, first %r: %r vs %r" % (
            what, k, len(bad), tuple(bad[0]), g[tuple(bad[0])], ref[tuple(bad[0])])


class Pair:
    """A BatchedAnts batch and one Q14Oracle per env, driven together; every output and the whole state compared
    after every call."""

    def __init__(self, cfg, worlds, record="compact8", evap_mode="lazy", rng_seed=9):
        from antsrl_b200 import BatchedAnts
        import torch
        self.torch, self.cfg, self.record, self.seed = torch, cfg, record, rng_seed
        self.E = len(worlds)
        self.o = [Q14Oracle(cfg, w) for w in worlds]
        self.b = BatchedAnts(cfg, self.E, evap_mode=evap_mode, record=record, rng_seed=rng_seed)
        self.b.import_state(stack_init(cfg, worlds))
        self.check("import")

    def close(self):
        self.b.close()

    def check(self, what):
        st = self.b.export_state()
        compare_state(st, self.o, what, self.cfg)
        strict_check(st, self.o, what, self.record)

    def observe(self):
        obs, ast, st, rew = self.b.observe()
        refs = []
        for o in self.o:
            p_, a_, s_ = o.observation()
            refs.append((p_, a_, o.s["rewards"].copy(), s_))
        check_outputs(self.cfg, (obs, ast, rew, st), refs, "observe")
        self.check("after observe")

    def activate(self):
        acts = activations(self.cfg, np.stack([o.s["activation"] for o in self.o]))
        for o, a in zip(self.o, acts):
            o.activate_all_pheromones(a)
        self.b.activate_all_pheromones(acts)

    def step(self, rot, ph, what):
        t = self.torch
        refs = [o.step(None if rot is None else rot[e].astype(np.int64), None if ph is None else ph[e].astype(np.int64))
                for e, o in enumerate(self.o)]
        out = self.b.step(None if rot is None else t.from_numpy(rot).cuda(), None if ph is None else t.from_numpy(ph).cuda())
        check_outputs(self.cfg, out[:3], [(r[0], r[1], r[2].copy()) for r in refs], what)
        self.check("after " + what)

    def update(self, noise, what):
        for e, o in enumerate(self.o):
            o.update(noise[e] if noise is not None else philox_uniform(self.seed, e, int(o.s["timestep"]), self.cfg["n_ants"]))
        self.b.update(None if noise is None else self.torch.from_numpy(noise).cuda())
        self.check("after " + what)


def run_loop(cfg, worlds, record="compact8", evap_mode="lazy", T=4):
    """import; observe; activate_all_pheromones; T x [step; update] on the tapes: every call compared."""
    pr = Pair(cfg, worlds, record, evap_mode)
    try:
        rot, rot_none, ph, ph_none, noise = tapes(cfg, worlds, T)
        pr.observe()
        pr.activate()
        for t in range(T):
            pr.step(None if rot_none[t] else rot[t], None if ph_none[t] else ph[t], "step %d" % t)
            pr.update(noise[t], "update %d" % t)
    finally:
        pr.close()


def worlds_of(name):
    cfg, E = batch_cfg(name)
    return cfg, [step_world(cfg, e) for e in range(E)]


FUSED = [(n, rec) for n in ("n11", "n300", "n1000") for rec in ("compact8", "compact", "f64")]


@pytest.mark.gpu
@pytest.mark.parametrize("name,rec", FUSED, ids=["%s-%s" % c for c in FUSED])
def test_step_update_loop_fused(name, rec):
    """k_env<0,1> and <1,0>: 23 envs per block with a partial last block (N = 11), 512 x 1 (N = 300), 512 x 2 (1000)."""
    run_loop(*worlds_of(name), record=rec)


@pytest.mark.gpu
@pytest.mark.parametrize("tpb", ("256", "1024"))
def test_fused_1024_ant_block_shapes(tpb, monkeypatch):
    """The 1024-ant block as 256 threads x 4 ants and 1024 x 1."""
    monkeypatch.setenv("ANTS_ENV_TPB", tpb)
    run_loop(*worlds_of("n1000"), record="compact8")


@pytest.mark.gpu
@pytest.mark.parametrize("path", ("fused", "flat"))
@pytest.mark.parametrize("mode", range(5))
def test_mandible_rule_modes(mode, path, monkeypatch):
    if path == "flat":
        monkeypatch.setenv("ANTS_NO_FUSED", "1")
    run_loop(*worlds_of("mode%d" % mode), record="compact8")


FLAT = [("n11", "compact8", "lazy"), ("n11", "f64", "lazy"), ("n1030", "compact8", "lazy"), ("n1030", "f64", "lazy"),
        ("n11", "f64", "dense"), ("n11", "f64", "tiles")]


@pytest.mark.gpu
@pytest.mark.parametrize("name,rec,evap", FLAT, ids=["%s-%s-%s" % c for c in FLAT])
def test_step_update_loop_flat(name, rec, evap, monkeypatch):
    """The flat kernels: ANTS_NO_FUSED, more than 1024 ants per env, the eager fields."""
    monkeypatch.setenv("ANTS_NO_FUSED", "1")
    run_loop(*worlds_of(name), record=rec, evap_mode=evap)


@pytest.mark.gpu
def test_step_update_loop_diffusion():
    """Pheromone diffusion (f64 planes carrying the wall bit in their sign): a deposit on a wall cell."""
    cfg = step_cfg(11, n_rocks=64, diffuse_factor=0.02, evap_factor=0.01)
    run_loop(cfg, [step_world(cfg, e) for e in range(50)], record="f64", evap_mode="dense")


@pytest.mark.gpu
@pytest.mark.parametrize("rec", ("compact8", "f64"))
def test_tiny_map(rec):
    cfg = tiny_cfg()
    run_loop(cfg, [step_world(cfg, e) for e in range(4)], record=rec)


@pytest.mark.gpu
@pytest.mark.parametrize("groups", ("1", "3"))
def test_rollout(groups, monkeypatch):
    """ants_rollout (<1,1> between the steps; with 3 groups on streams of their own) with Philox noise: the last step's
    outputs and the state equal the oracle."""
    import torch
    from antsrl_b200 import BatchedAnts
    monkeypatch.setenv("ANTS_ROLLOUT_GROUPS", groups)
    cfg, worlds = worlds_of("n11")
    E, T, seed = len(worlds), 4, 9
    rot, _, ph, _, _ = tapes(cfg, worlds, T)
    b = BatchedAnts(cfg, E, evap_mode="lazy", record="compact8", rng_seed=seed)
    try:
        b.import_state(stack_init(cfg, worlds))
        b.observe()
        out = b.rollout(torch.from_numpy(rot).cuda().contiguous(), torch.from_numpy(ph).cuda().contiguous())
        oracles = [Q14Oracle(cfg, w) for w in worlds]
        refs = []
        for e, o in enumerate(oracles):
            o.observation()
            for t in range(T):
                r = o.step(rot[t, e].astype(np.int64), ph[t, e].astype(np.int64))
                o.update(philox_uniform(seed, e, int(o.s["timestep"]), cfg["n_ants"]))
            refs.append((r[0], r[1], r[2].copy()))
        check_outputs(cfg, out, refs, "last step of the rollout")
        st = b.export_state()
        compare_state(st, oracles, "after the rollout", cfg)
        strict_check(st, oracles, "after the rollout", "compact8")
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ("fused", "flat"))
def test_import_then_update(path, monkeypatch):
    """The first update after an import reads the wall bit from the record (no move wrote the flag)."""
    if path == "flat":
        monkeypatch.setenv("ANTS_NO_FUSED", "1")
    cfg, worlds = worlds_of("n11")
    pr = Pair(cfg, worlds)
    try:
        rot, _, ph, _, noise = tapes(cfg, worlds, 2)
        pr.update(noise[0], "update 0")
        assert sum(o.ev["wall_hit_record"] for o in pr.o) > 0
        pr.step(rot[1], ph[1], "step 1")
        pr.update(noise[1], "update 1")
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ("fused", "flat"))
def test_two_steps_without_an_update(path, monkeypatch):
    """import -> step -> step -> update: the move without an update stamps every ant (all_stamp), the update takes the
    queue of two steps."""
    if path == "flat":
        monkeypatch.setenv("ANTS_NO_FUSED", "1")
    cfg, worlds = worlds_of("n11")
    pr = Pair(cfg, worlds)
    try:
        rot, _, ph, _, noise = tapes(cfg, worlds, 3)
        pr.observe()
        pr.step(None, None, "step 0")
        pr.step(rot[1], ph[1], "step 1")
        pr.update(noise[1], "update")
        pr.step(rot[2], ph[2], "step 2")
        pr.update(noise[2], "update 2")
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ("fused", "flat"))
@pytest.mark.parametrize("rec", ("compact8", "f64"))
def test_queue_overflow(rec, path, monkeypatch):
    """D2: two steps without an update queue 2 E N cells, more than the flat kernels' batch-wide list (E N pairs)
    and more than an env's segment of the fused one (N): both must sweep the discs instead."""
    if path == "flat":
        monkeypatch.setenv("ANTS_NO_FUSED", "1")
    cfg = step_cfg(40, mode=3)
    worlds = [overflow_world(cfg, e) for e in range(5)]
    pr = Pair(cfg, worlds, record=rec)
    try:
        pr.observe()
        pr.step(None, None, "step 0")
        pr.step(None, None, "step 1")
        assert sum(o.queued for o in pr.o) > pr.E * cfg["n_ants"]
        pr.update(np.full((pr.E, cfg["n_ants"]), 0.5), "update")
        pr.step(None, None, "step 2")
        pr.update(None, "update 2")
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ("fused", "flat"))
@pytest.mark.parametrize("how", ("import", "generate"))
def test_window_episode_between_step_and_update(how, path, monkeypatch):
    """D1: a step queues drops inside the disc of every env; envs [1, 3) then start a new episode (a windowed import,
    or ants_generate_env_maps for the window) whose disc lies elsewhere and whose food covers the queued cells.  The
    update must leave that food alone (the reference's Anthill.update only sees the new disc)."""
    if path == "flat":
        monkeypatch.setenv("ANTS_NO_FUSED", "1")
    cfg, worlds = worlds_of("n11")
    pr = Pair(cfg, worlds)
    try:
        rot, _, ph, _, noise = tapes(cfg, worlds, 3)
        pr.observe()
        pr.step(None, None, "step 0")
        assert all(o.queued >= 2 for o in pr.o[1:3])
        ts, alias = int(pr.o[0].s["timestep"]), pr.o[0].s["rw_alias"]
        if how == "import":
            new = [step_world(cfg, 100 + e, hill=ALT_HILL, old_hill=HILL) for e in (1, 2)]
            st = stack_init(cfg, new)
            for k in ("act_bool", "rw_alias", "timestep"):
                st.pop(k, None)
            pr.b.import_state(st, envs=(1, 2))
            for e, w in zip((1, 2), new):
                o = Q14Oracle(cfg, dict(w, rw_prev_dist=st["rw_prev_dist"][e - 1]))
                o.s["timestep"], o.s["rw_alias"], o.s["act_bool"] = ts, alias, pr.o[e].s["act_bool"]
                pr.o[e] = o
        else:
            food_discs = np.array([[[2, 1, 1], [1, 4, 1]]] * 2, np.int32)      # over the queued cells (2, 1), (0, 4)
            wall_discs = np.array([[[30, 10, 2]]] * 2, np.int32)
            pr.b.generate_env_maps(np.array([ALT_HILL] * 2, np.int32), wall_discs, food_discs, envs=(1, 2))
            maps = pr.b.export_state(keys=("food", "walls", "phero", "explored", "anthill_xyr"), envs=(1, 2))
            for k, e in enumerate((1, 2)):
                o = pr.o[e]
                for key in ("food", "walls", "phero", "explored", "anthill_xyr"):
                    o.s[key] = maps[key][k].copy()
                assert o.s["food"][2, 1] > 0 and o.s["food"][0, 4] > 0
                o.area = anthill_area(cfg["w"], cfg["h"], *[int(v) for v in o.s["anthill_xyr"]])
        for e in (1, 2):
            assert not pr.o[e].area[2, 1] and not pr.o[e].area[0, 4]
        pr.check("after the new episode of envs 1, 2")
        pr.update(noise[0], "update 0")
        pr.step(rot[1], ph[1], "step 1")
        pr.update(noise[1], "update 1")
    finally:
        pr.close()
