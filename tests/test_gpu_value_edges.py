"""Values at their edges: activations and imported fields against the oracle, non-finite inputs refused.

The caller controls three kinds of float values: the activations (ants_activate_all_pheromones after
agent.initialize, or `activation` in an import) and the imported pheromone and food planes.  `value_world` builds one
env's complete state whose ants stand still (max_speed 0) on chosen cells, so that on chosen updates:
  * activations of -0.75, -300, -0.0, +-5e-324, 0.005 (below the cut), exactly max_val on an empty cell, values that
    land the sum on a saturated deposit exactly on max_val and one double either side of it, and 1e300;
  * those deposits land on an empty cell, a plain value, a boxed (saturated) deposit, a wall cell and a cell imported
    negative;
  * imported pheromone: negative, -0.0, subnormal, max_val and max_val -+ 1 ulp, 255.2 (v * 0.999 < 255) and 255.3
    (v * 0.999 > 255), 300, 1000, a value below the cut (the values above max_val only where they are accepted: the
    eager modes, and runs without max_val);
  * imported food: a negative integer, a negative non-integer, -0.0, negative food under ants whose mandibles stay
    closed and under one that opens and drops onto it, negative food inside the anthill disc (absorbed into
    anthill_food).
The same worlds run with bool activations and without max_val (the oracle's phero_max_val = None; no pheromone
channel then, RL_api.py:125 divides by max_val).  The CPU tests replay every batch on the oracle and assert that each
class occurs, and show that a NaN or -inf activation and a NaN import spread NaN through the reference's convolution
(the reason those inputs are refused instead of emulated).  The GPU tests compare every output and the whole state
after every call, in every record format and evaporation mode, on the block-per-env kernels, the flat ones, ants_rollout
and the generic perception kernel, check that negative integer food is the one thing that keeps an observation off the
packed transport, and check what ants_activate_all_pheromones and ants_import_env_state refuse."""
from collections import Counter

import numpy as np
import pytest
from scipy.signal import convolve2d

from oracle.antsrl_oracle import OracleEnv, make_config, philox_uniform
from parity_util import compare_state, stack_init
from test_gpu_perception_edges import check_outputs
from test_gpu_step_edges import strict_check

MAX = 255.0
CUT = 0.01
W, H, N, P = 40, 35, 16, 2
HILL = (30, 25, 3)
CHANNELS = ["ants", "phero0", "phero1", "food", "walls", "anthill"]   # mandible rule (m | f) & !h
NOISE = 0.5                                                          # theta += 0 for the ant standing in a wall
T_LOOP = 4
E = 5


def below(v):
    return float(np.nextafter(v, -np.inf))


def above(v):
    return float(np.nextafter(v, np.inf))


def value_cfg(max_val=MAX, n_rocks=0, **kw):
    ch = CHANNELS if max_val is not None else [c for c in CHANNELS if not c.startswith("phero")]
    if n_rocks:
        ch = ch + ["rocks"]
    return make_config(W, H, N, n_phero=P, n_rocks=n_rocks, channels=ch, fwd_delta=0, max_speed=0.0,
                       max_time=100000, phero_max_val=max_val, **kw)


def landing(target, base):
    """a with fl(base + a) == target, the doubles around target - base walked outward."""
    lo = hi = target - base
    for _ in range(64):
        for a in (lo, hi):
            if base + a == target:
                return float(a)
        lo, hi = below(lo), above(hi)
    raise AssertionError("no double a with %r + a == %r" % (base, target))


def keep(cfg):
    """The centre tap of the update's convolution (DIFFUSE_FACTOR 0): value * keep is one update's evaporation."""
    return (1.0 - 8.0 * cfg["diffuse_factor"]) * (1.0 - cfg["evap_factor"])


# ------------------------------------------------------------------------------------------------ the worlds
def _ants(cfg):
    """(cell, what the cell holds, activations, food, holding, mandibles) of the 16 ants."""
    m = MAX if cfg["phero_max_val"] is None else cfg["phero_max_val"]
    e = m * keep(cfg)                       # a saturated deposit after one update (decay_table[1])
    return [((4, 5), "empty", (-0.75, m), 0.0, 0.0, 0),
            ((8, 5), "plain", (-300.0, 0.005), 0.0, 0.0, 0),
            ((12, 5), "boxed", (1e300, -0.75), 0.0, 0.0, 0),
            ((16, 5), "wall", (0.75, -0.75), 0.0, 0.0, 0),
            ((20, 5), "negative", (0.75, 5e-324), 0.0, 0.0, 0),
            ((24, 5), "empty", (-0.0, -5e-324), 0.0, 0.0, 0),
            ((28, 5), "plain", (1e300, -0.0), 0.0, 0.0, 0),
            ((32, 5), "boxed", (-300.0, 0.75), 0.0, 0.0, 0),
            ((4, 10), "boxed", (landing(m, e), landing(below(m), e)), 0.0, 0.0, 0),
            ((8, 10), "boxed", (landing(above(m), e), 0.005), 0.0, 0.0, 0),
            ((12, 10), "empty", (5e-324, m), 0.0, 0.0, 0),
            ((16, 10), "plain", (-0.0, 0.75), 0.0, 0.0, 0),
            ((6, 20), "empty", (0.75, 0.0), -3.0, 2.0, 1),        # closed over negative food: stays closed
            ((29, 25), "empty", (0.0, 0.75), -2.5, 2.0, 1),       # in the hill: opens, drops 2 onto -2.5
            ((31, 25), "empty", (0.75, 0.0), -0.0, 0.0, 0),
            ((10, 20), "empty", (0.0, -0.75), -2.5, 0.0, 0)]


def imported_values(cfg, eager):
    """The imported pheromone values of the row y = 30; those above max_val only where an import accepts them."""
    m = MAX if cfg["phero_max_val"] is None else cfg["phero_max_val"]
    vals = [-7.5, -0.0, 5e-324, 2.2e-308, m, below(m), 0.005, 0.5]
    if eager or cfg["phero_max_val"] is None:
        vals += [above(m), 255.2, 255.3, 300.0, 1000.0]
    return vals


FOOD = {(2, 33): -3.0, (4, 33): -2.5, (6, 33): -0.0, (8, 33): 7.0,
        (30, 27): -4.0, (28, 24): -1.25, (32, 26): 3.0, (30, 23): -0.0}      # (the last four in the disc)


def value_world(cfg, seed, eager=False):
    """One env's complete state (OracleEnv / stack_init schema).  `eager`: the import may hold values above max_val."""
    rng = np.random.RandomState(800 + seed)
    m = MAX if cfg["phero_max_val"] is None else cfg["phero_max_val"]
    ants = _ants(cfg)
    phero = np.zeros((P, W, H))
    walls = np.zeros((W, H), bool)
    food = np.zeros((W, H))
    for (cx, cy), what, _, f, _, _ in ants:
        if what == "plain":
            phero[:, cx, cy] = (100.0, 37.5)
        elif what == "boxed":
            phero[:, cx, cy] = m
        elif what == "negative":
            phero[:, cx, cy] = (-3.0, -0.5)
        elif what == "wall":
            walls[cx, cy] = True
            phero[:, cx, cy] = 7.0
        food[cx, cy] = f
    for (cx, cy), f in FOOD.items():
        food[cx, cy] = f
    for j, v in enumerate(imported_values(cfg, eager)):
        phero[j % P, 2 + 2 * j, 30] = v
        phero[(j + 1) % P, 3 + 2 * j, 31] = v
    for x in range(2, 38, 3):                       # env-specific plain values and food, away from the ants
        phero[x % P, x, 15] = rng.uniform(0.02, 200.0)
        food[x, 17] = float(rng.randint(0, 4))
    cells = [c for c, *_ in ants]
    x = np.array([cx + 0.375 for cx, _ in cells])
    y = np.array([cy + 0.625 for _, cy in cells])
    theta = rng.uniform(0, 2 * np.pi, N)
    world = {"x": x, "y": y, "theta": theta, "prev_x": x.copy(), "prev_y": y.copy(), "prev_theta": theta.copy(),
             "holding": np.array([a[4] for a in ants]),
             "mandibles": np.array([a[5] for a in ants], np.uint8), "reward_state": np.zeros(N, np.uint8),
             "seed": rng.random_sample(N), "activation": np.array([a[2] for a in ants]),
             "rw_holding_prev": np.zeros(N), "rewards": np.zeros(N), "walls": walls.astype(np.uint8), "food": food,
             "phero": phero, "explored": np.zeros((W, H), np.uint8), "anthill_xyr": np.array(HILL, np.int32),
             "anthill_food": np.float64(seed), "act_bool": False}
    if cfg["n_rocks"]:
        world.update(rock_centers=np.array([[36.5, 30.5], [2.5, 26.5]][:cfg["n_rocks"]]),
                     rock_radii=np.full(cfg["n_rocks"], 1.0), rock_weights=np.full(cfg["n_rocks"], 50.0))
    return world


def clean_world(world, cfg):
    """The world without negative, -0.0 or above-max values (what diffusion and every mode accept)."""
    w = dict(world)
    m = MAX if cfg["phero_max_val"] is None else cfg["phero_max_val"]
    w["phero"] = np.minimum(np.abs(world["phero"]), m)
    w["food"] = np.abs(world["food"])
    w["activation"] = np.minimum(np.abs(world["activation"]), m)
    return w


# ------------------------------------------------------------------------------------------------ the oracle
class ValueOracle(OracleEnv):
    """OracleEnv whose step and update count the classes this file builds in `ev`."""

    def __init__(self, cfg, state):
        super().__init__(cfg, state)
        self.ev = Counter()
        s, ev = self.s, self.ev
        m = cfg["phero_max_val"]
        f, ph = s["food"], s["phero"]
        neg = f < 0
        ev["food_neg_int"] += int((neg & (f == np.floor(f))).sum())
        ev["food_neg_frac"] += int((neg & (f != np.floor(f))).sum())
        ev["food_minus_zero"] += int(((f == 0) & np.signbit(f)).sum())
        ev["food_neg_in_hill"] += int((neg & self.area).sum())
        ev["phero_neg"] += int((ph < 0).sum())
        ev["phero_minus_zero"] += int(((ph == 0) & np.signbit(ph)).sum())
        ev["phero_subnormal"] += int(((ph != 0) & (np.abs(ph) < np.finfo(float).tiny)).sum())
        ev["phero_below_cut"] += int(((ph > 0) & (ph * keep(cfg) < CUT)).sum())
        mv = MAX if m is None else m
        ev["phero_at_max"] += int((ph == mv).sum())
        ev["phero_max_minus_ulp"] += int((ph == below(mv)).sum())
        ev["phero_max_plus_ulp"] += int((ph == above(mv)).sum())
        ev["phero_above_clamped_at_1"] += int(((ph > mv) & (ph * keep(cfg) > mv)).sum())
        ev["phero_above_evaporated_below"] += int(((ph > mv) & (ph * keep(cfg) < mv)).sum())
        ev["phero_300_1000"] += int(((ph == 300.0) | (ph == 1000.0)).sum())

    def step(self, rotation, pheromone):
        s, ev = self.s, self.ev
        pcx, pcy = s["prev_x"].astype(int), s["prev_y"].astype(int)
        f = s["food"][pcx, pcy]
        old = s["mandibles"].copy()
        out = super().step(rotation, pheromone)
        new = s["mandibles"]
        ev["closed_over_negative_food"] += int(((old == 1) & (new == 1) & (f < 0)).sum())
        ev["drop_onto_negative_food"] += int(((old == 1) & (new == 0) & (f < 0) & (s["holding"] == 0)).sum())
        return out

    def update(self, noise=None):
        s, cfg, ev = self.s, self.cfg, self.ev
        m = cfg["phero_max_val"]
        mv = MAX if m is None else m
        walls = s["walls"].astype(bool)
        before = s["phero"].copy()
        ev["negative_food_absorbed"] += int(((s["food"] < 0) & self.area).sum())
        ph = before.copy()
        ph[:, walls] = 0
        evap = np.stack([convolve2d(p, self.filter, 'same', 'fill', 0) for p in ph])
        evap[evap < CUT] = 0
        # the deposits of the update (last ant wins), classified by activation and by what lies on the cell
        cx, cy = s["x"].astype(int), s["y"].astype(int)
        last = np.full(W * H, -1)
        last[cx * H + cy] = np.arange(N)
        own = last[cx * H + cy] == np.arange(N)
        for k in range(P):
            a = s["activation"][:, k]
            dep = own & (a != 0)
            b, e = before[k][cx, cy], evap[k][cx, cy]
            on = np.where(walls[cx, cy], "wall", np.where(b < 0, "negative", np.where(
                b == 0, "empty", np.where(b == mv, "boxed", "plain"))))
            for j in np.flatnonzero(dep):
                ev["deposit_on_" + on[j]] += 1
            ev["act_neg"] += int((dep & (a < 0) & (a > -1)).sum())
            ev["act_neg_300"] += int((dep & (a == -300.0)).sum())
            ev["act_minus_zero"] += int((own & (a == 0) & np.signbit(a)).sum())
            ev["act_min_subnormal"] += int((dep & (a == 5e-324)).sum())
            ev["act_neg_min_subnormal"] += int((dep & (a == -5e-324)).sum())
            ev["act_below_cut"] += int((dep & (a == 0.005)).sum())
            ev["act_max_on_empty"] += int((dep & (a == mv) & (b == 0)).sum())
            ev["act_1e300"] += int((dep & (a == 1e300)).sum())
            ev["act_1"] += int((dep & (a == 1.0)).sum())
            if m is not None:
                ev["sum_at_max"] += int((dep & (e + a == m) & (a != m)).sum())
                ev["sum_below_max"] += int((dep & (e + a == below(m))).sum())
                ev["sum_above_max"] += int((dep & (e + a == above(m))).sum())
        super().update(noise)


REQUIRED = ["food_neg_int", "food_neg_frac", "food_minus_zero", "food_neg_in_hill", "phero_neg", "phero_minus_zero",
            "phero_subnormal", "phero_below_cut", "phero_at_max", "phero_max_minus_ulp", "closed_over_negative_food",
            "drop_onto_negative_food", "negative_food_absorbed", "deposit_on_wall", "deposit_on_negative",
            "deposit_on_empty", "deposit_on_plain", "deposit_on_boxed"]
FLOAT_ACTS = ["act_neg", "act_neg_300", "act_minus_zero", "act_min_subnormal", "act_neg_min_subnormal",
              "act_below_cut", "act_max_on_empty", "act_1e300"]
ABOVE_MAX = ["phero_max_plus_ulp", "phero_above_clamped_at_1", "phero_above_evaporated_below", "phero_300_1000"]


# ------------------------------------------------------------------------------------------------ batches
# (record, evap_mode): the record formats and evaporation modes of the GPU tests
LAYOUTS = [("f64", "lazy"), ("compact", "lazy"), ("compact8", "lazy"), ("f64", "dense"), ("f64", "tiles")]


def batch(max_val=MAX, evap="lazy", n=E):
    cfg = value_cfg(max_val)
    return cfg, [value_world(cfg, e, eager=evap != "lazy") for e in range(n)]


def activations(worlds, as_bool=False):
    act = np.stack([w["activation"] for w in worlds])
    return act != 0 if as_bool else act


def replay(cfg, worlds, T, as_bool=False, noise=None):
    """observe; activate_all_pheromones; T x [step (None actions); update] on ValueOracle: the summed counts."""
    oracles = [ValueOracle(cfg, w) for w in worlds]
    act = activations(worlds, as_bool)
    for e, o in enumerate(oracles):
        o.observation()
        o.activate_all_pheromones(act[e])
        for t in range(T):
            o.step(None, None)
            o.update(np.full(N, NOISE) if noise is None else noise(e, o))
    ev = Counter()
    for o in oracles:
        ev.update(o.ev)
    return ev


def required(cfg, evap, as_bool=False):
    keys = list(REQUIRED) + (["act_1"] if as_bool else FLOAT_ACTS)
    if cfg["phero_max_val"] is not None and not as_bool:
        keys += ["sum_at_max", "sum_below_max", "sum_above_max"]
    if evap != "lazy" or cfg["phero_max_val"] is None:
        keys += ABOVE_MAX
    return keys


CPU_RUNS = [(MAX, "lazy", False), (MAX, "dense", False), (None, "lazy", False), (None, "dense", False),
            (MAX, "lazy", True)]


@pytest.mark.parametrize("max_val,evap,as_bool", CPU_RUNS)
def test_value_worlds_cover_every_class(max_val, evap, as_bool):
    cfg, worlds = batch(max_val, evap)
    ev = replay(cfg, worlds, T_LOOP, as_bool)
    missing = [k for k in required(cfg, evap, as_bool) if ev[k] == 0]
    assert not missing, "no %s; counts %r" % (missing, dict(ev))
    if evap == "lazy" and max_val is not None:
        assert ev["phero_max_plus_ulp"] == ev["phero_300_1000"] == 0, "a lazy import above max_val is refused"
    print(dict(sorted(ev.items())))


ROLLOUT_SEED = 11
PACKED_STEPS = 3
ROLLOUTS = [("compact8", 4), ("f64", 4), ("compact8", 270)]


def philox_noise(e, o):
    return philox_uniform(ROLLOUT_SEED, e, int(o.s["timestep"]), N)


@pytest.mark.parametrize("T", sorted({t for _, t in ROLLOUTS}))
def test_rollout_worlds_cover_every_class(T):
    """The rollouts of test_values_rollout (Philox collision noise, T updates) on the oracle."""
    cfg, worlds = batch(MAX, "lazy")
    ev = replay(cfg, worlds, T, noise=philox_noise)
    missing = [k for k in required(cfg, "lazy") if ev[k] == 0]
    assert not missing, "T = %d: no %s; counts %r" % (T, missing, dict(ev))


def test_refusal_worlds_are_accepted_everywhere():
    """The worlds of the refusal tests (two rocks, diffusion factors in one mode) hold nothing any mode refuses -- no
    negative, -0.0, non-finite or above-max value -- so each refusal comes from the one value a test puts in; and
    their loop still deposits onto empty, plain, saturated and wall cells."""
    for _, evap in MODES:
        cfg = refusal_cfg(evap)
        worlds = refusal_worlds(cfg)
        for w in worlds:
            for k in ("phero", "food", "activation", "x", "y", "theta", "holding", "rock_centers", "rock_radii",
                      "rock_weights"):
                v = np.asarray(w[k], float)
                assert np.isfinite(v).all() and not np.signbit(v).any(), (evap, k)
            assert w["phero"].max() <= MAX and w["activation"].max() <= MAX, evap
        ev = replay(cfg, worlds, 1)
        for k in ("deposit_on_empty", "deposit_on_plain", "deposit_on_boxed", "deposit_on_wall"):
            assert ev[k] > 0, (evap, k, dict(ev))


def packed_world(cfg, e, negative):
    """value_world with integer food only: -2.5 -> -2, -1.25 -> -1 (the drop of 2 onto -2 leaves 0), and with
    `negative` False every amount made non-negative.  The packed transport (k_pack_obs) takes integer food in
    [0, 65535); here a negative sign is the only reason a sample has no packed form."""
    w = value_world(cfg, e)
    w["food"] = np.trunc(w["food"]) if negative else np.abs(np.trunc(w["food"]))
    return w


def visible_food(cfg, perception):
    return perception[:, np.asarray(cfg["mask"], bool), cfg["channels"].index("food")]


@pytest.mark.parametrize("negative", (True, False))
def test_packed_worlds_hold_integer_food_in_view(negative):
    """Every food sample an ant sees in the steps of test_negative_food_packed_falls_back is an integer below 65535;
    in the negative worlds some are negative on every step, in the control worlds none is."""
    cfg = value_cfg()
    oracles = [OracleEnv(cfg, packed_world(cfg, e, negative)) for e in range(E)]
    for o in oracles:
        o.observation()
        o.activate_all_pheromones(o.s["activation"])
    for t in range(PACKED_STEPS):
        f = np.concatenate([visible_food(cfg, o.step(None, None)[0]) for o in oracles])
        assert (f == np.floor(f)).all() and (f < 65535).all(), "step %d" % t
        assert ((f < 0).sum() > 0) == negative, "step %d: %d negative samples" % (t, (f < 0).sum())
        for o in oracles:
            o.update(np.full(N, NOISE))


def nan_cells_per_update(cfg, world, T=3):
    o = OracleEnv(cfg, world)
    counts = []
    for _ in range(T):
        o.update(np.full(N, NOISE))
        counts.append(int(np.isnan(o.s["phero"]).sum()))
    return counts


@pytest.mark.parametrize("how", ("nan_activation", "minus_inf_activation", "nan_import"))
def test_reference_spreads_nan(how):
    """The reference's convolution multiplies the zero ring taps by a NaN (or the -inf of a deposit): one such cell
    is more NaN cells after each update -- which is why the kernels refuse these inputs rather than emulate them."""
    cfg = value_cfg()
    w = clean_world(value_world(cfg, 0), cfg)
    w["activation"] = np.zeros((N, P))
    if how == "nan_import":
        w["phero"][0, 20, 20] = np.nan
    else:
        w["activation"][0, 0] = np.nan if how == "nan_activation" else -np.inf
    counts = nan_cells_per_update(cfg, w)
    # (a -inf deposit is -inf after its update; its 8 neighbours are NaN after the next one)
    assert 0 < counts[1] < counts[2] and counts[0] <= counts[1], counts
    print(how, counts)


# ------------------------------------------------------------------------------------------------ GPU
class ValuePair:
    """A BatchedAnts batch and one ValueOracle per env, driven together; every output and the whole state compared
    after every call."""

    def __init__(self, cfg, worlds, record, evap_mode, as_bool=False, rng_seed=11):
        from antsrl_b200 import BatchedAnts
        import torch
        self.torch, self.cfg, self.record, self.seed = torch, cfg, record, rng_seed
        self.E = len(worlds)
        self.act = activations(worlds, as_bool)
        self.o = [ValueOracle(cfg, w) for w in worlds]
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
        for o, a in zip(self.o, self.act):
            o.activate_all_pheromones(a)
        self.b.activate_all_pheromones(self.act)
        self.check("after activate_all_pheromones")

    def step(self, what):
        refs = [o.step(None, None) for o in self.o]
        out = self.b.step(None, None)
        check_outputs(self.cfg, out[:3], [(r[0], r[1], r[2].copy()) for r in refs], what)
        self.check("after " + what)

    def update(self, what):
        for o in self.o:
            o.update(np.full(self.cfg["n_ants"], NOISE))
        self.b.update(self.torch.full((self.E, self.cfg["n_ants"]), NOISE, dtype=self.torch.float64, device="cuda"))
        self.check("after " + what)

    def rollout(self, T):
        """ants_rollout with None actions (the activations stay) and Philox noise; the last step's outputs and the
        state compared."""
        out = self.b.rollout(None, None, n_steps=T)
        refs = []
        for e, o in enumerate(self.o):
            for _ in range(T):
                r = o.step(None, None)
                o.update(philox_uniform(self.seed, e, int(o.s["timestep"]), self.cfg["n_ants"]))
            refs.append((r[0], r[1], r[2].copy()))
        check_outputs(self.cfg, out, refs, "last step of a rollout of %d" % T)
        self.check("after a rollout of %d" % T)


def run_loop(cfg, worlds, record, evap_mode, as_bool=False, T=T_LOOP):
    """import; observe; activate_all_pheromones; T x [step; update]: every call compared."""
    pr = ValuePair(cfg, worlds, record, evap_mode, as_bool)
    try:
        pr.observe()
        pr.activate()
        for t in range(1, T + 1):
            pr.step("step %d" % t)
            pr.update("update %d" % t)
        return pr.o
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("record,evap", LAYOUTS, ids=["%s-%s" % c for c in LAYOUTS])
def test_values_fused(record, evap):
    """The block-per-env kernels and the row perception kernel in every record format and evaporation mode."""
    cfg, worlds = batch(MAX, evap)
    oracles = run_loop(cfg, worlds, record, evap)
    ev = Counter()
    for o in oracles:
        ev.update(o.ev)
    assert not [k for k in required(cfg, evap) if ev[k] == 0], dict(ev)


FLAT = [("compact8", "lazy"), ("f64", "lazy"), ("f64", "dense")]


@pytest.mark.gpu
@pytest.mark.parametrize("record,evap", FLAT, ids=["%s-%s" % c for c in FLAT])
def test_values_flat(record, evap, monkeypatch):
    monkeypatch.setenv("ANTS_NO_FUSED", "1")
    run_loop(*batch(MAX, evap), record, evap)


@pytest.mark.gpu
def test_values_generic_perception(monkeypatch):
    monkeypatch.setenv("ANTS_PERCEIVE_GENERIC", "1")
    run_loop(*batch(MAX, "lazy"), "compact8", "lazy")


NO_MAX = [("f64", "lazy"), ("f64", "dense"), ("f64", "tiles")]


@pytest.mark.gpu
@pytest.mark.parametrize("record,evap", NO_MAX, ids=["%s-%s" % c for c in NO_MAX])
def test_values_without_max_val(record, evap):
    """phero_max_val None: no clamp; 1e300 deposits and imports above 255 kept as they are.  (The f32 values of the
    compact records cannot hold 1e300: DESIGN section 4.)"""
    run_loop(*batch(None, evap), record, evap)


@pytest.mark.gpu
@pytest.mark.parametrize("record", ("compact8", "f64"))
def test_values_bool_activations(record):
    run_loop(*batch(MAX, "lazy"), record, "lazy", as_bool=True)


@pytest.mark.gpu
@pytest.mark.parametrize("record,T", ROLLOUTS)
def test_values_rollout(record, T):
    """ants_rollout; with T = 270 the compact8 plain values (negative deposits, escaped negative food) cross the
    8-bit timestamp fold (k_lazy_fold)."""
    cfg, worlds = batch(MAX, "lazy")
    pr = ValuePair(cfg, worlds, record, "lazy", rng_seed=ROLLOUT_SEED)
    try:
        pr.observe()
        pr.activate()
        pr.rollout(T)
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("negative", (True, False), ids=("negative", "control"))
def test_negative_food_has_no_packed_form(negative, monkeypatch):
    """k_pack_obs packs integer food in [0, 65535).  packed_world holds integer food only, negative amounts in the
    negative worlds: there, and only there, ants_step_host_packed reports on every step that the observation has no
    packed form (ANTS_E_STATE, the step taken), and ants_step_host with the packed transport forced falls back to the
    dense copy.  In both worlds ants_step_host's observation (expanded from the packed form in the control worlds)
    equals the device step's bit for bit and the oracle's."""
    import torch
    from antsrl_b200 import AntsError, BatchedAnts
    monkeypatch.setenv("ANTS_E2E_PACKED", "1")
    cfg = value_cfg()
    worlds = [packed_world(cfg, e, negative) for e in range(E)]
    oracles = [OracleEnv(cfg, w) for w in worlds]
    act = activations(worlds)
    hosts, packs, devs = [BatchedAnts(cfg, E, evap_mode="lazy", record="compact8") for _ in range(3)]
    try:
        for b in (hosts, packs, devs):
            b.import_state(stack_init(cfg, worlds))
            b.observe()
            b.activate_all_pheromones(act)
        for e, o in enumerate(oracles):
            o.observation()
            o.activate_all_pheromones(act[e])
        noise = np.full((E, N), NOISE)
        for t in range(PACKED_STEPS):
            refs = [o.step(None, None) for o in oracles]
            if negative:
                with pytest.raises(AntsError, match=r"no packed form .*code -3"):
                    packs.step_host_packed(None, None)
            else:
                packs.step_host_packed(None, None)
            h_obs, h_ast, h_rew, _ = hosts.step_host(None, None)
            d_obs, d_ast, d_rew, _ = devs.step(None, None)
            assert np.array_equal(h_obs, d_obs.cpu().numpy()), "step %d: the host observation differs" % t
            assert np.array_equal(h_ast, d_ast.cpu().numpy()) and np.array_equal(h_rew, d_rew.cpu().numpy())
            check_outputs(cfg, (d_obs, d_ast, d_rew), [(r[0], r[1], r[2].copy()) for r in refs], "step %d" % t)
            for o, n in zip(oracles, noise):
                o.update(n)
            hosts.update_host(noise)
            for b in (packs, devs):
                b.update(torch.from_numpy(noise).cuda())
        for b in (hosts, packs):
            compare_state(b.export_state(), oracles, "after the host steps", cfg)
    finally:
        for b in (hosts, packs, devs):
            b.close()


# ------------------------------------------------------------------------------------------------ refusals
MODES = LAYOUTS + [("f64", "diffuse")]


def refusal_cfg(evap):
    kw = dict(diffuse_factor=0.02, evap_factor=0.01) if evap == "diffuse" else {}
    return value_cfg(MAX, n_rocks=2, **kw)


def refusal_worlds(cfg, E_=3):
    return [clean_world(value_world(cfg, e), cfg) for e in range(E_)]


def refusal_handle(record, evap):
    from antsrl_b200 import BatchedAnts
    cfg = refusal_cfg(evap)
    worlds = refusal_worlds(cfg)
    b = BatchedAnts(cfg, len(worlds), evap_mode="dense" if evap == "diffuse" else evap, record=record)
    b.import_state(stack_init(cfg, worlds))
    return cfg, worlds, b


def assert_unchanged(before, after, what):
    for k, v in before.items():
        assert np.array_equal(np.asarray(v), np.asarray(after[k])), "%s changed %s" % (what, k)


def run_on(cfg, worlds, b, what):
    """observe; activate; step; update on the handle and on fresh oracles of `worlds`: everything compared."""
    import torch
    oracles = [OracleEnv(cfg, w) for w in worlds]
    obs, ast, st, rew = b.observe()
    refs = []
    for o in oracles:
        p_, a_, s_ = o.observation()
        refs.append((p_, a_, o.s["rewards"].copy(), s_))
    check_outputs(cfg, (obs, ast, rew, st), refs, what + ": observe")
    act = activations(worlds)
    b.activate_all_pheromones(act)
    for o, a in zip(oracles, act):
        o.activate_all_pheromones(a)
    refs = [o.step(None, None) for o in oracles]
    out = b.step(None, None)
    check_outputs(cfg, out[:3], [(r[0], r[1], r[2].copy()) for r in refs], what + ": step")
    noise = np.full((len(worlds), N), NOISE)
    for o, n in zip(oracles, noise):
        o.update(n)
    b.update(torch.from_numpy(noise).cuda())
    compare_state(b.export_state(), oracles, what + ": update", cfg)


NON_FINITE = (float("nan"), float("inf"), float("-inf"))
ANT_KEYS = ("x", "y", "theta", "prev_x", "prev_y", "prev_theta", "holding")
ROCK_KEYS = ("rock_centers", "rock_radii", "rock_weights")


@pytest.mark.gpu
@pytest.mark.parametrize("record,evap", MODES, ids=["%s-%s" % c for c in MODES])
def test_non_finite_arrays_refused(record, evap):
    """NaN and +-inf activations (activate_all_pheromones, import_state) and per-ant and rock values: ANTS_E_ARG
    before anything is uploaded, the handle unchanged."""
    from antsrl_b200 import AntsError
    cfg, worlds, b = refusal_handle(record, evap)
    try:
        before = b.export_state()
        st = stack_init(cfg, worlds)
        for bad in NON_FINITE:
            act = activations(worlds)
            act[1, 3, 0] = bad
            with pytest.raises(AntsError):
                b.activate_all_pheromones(act)
            with pytest.raises(AntsError):
                b.import_state({"activation": act})
            with pytest.raises(AntsError):
                b.import_state({"activation": act[1:2]}, envs=(1, 1))
            for k in ANT_KEYS + ROCK_KEYS:
                v = np.array(st[k], copy=True)
                v.reshape(len(worlds), -1)[2, 1] = bad
                with pytest.raises(AntsError):
                    b.import_state({k: v})
                with pytest.raises(AntsError):     # with the other keys of a full import: none of them uploaded
                    b.import_state(dict(st, **{k: v}, phero=np.zeros_like(st["phero"])))
            assert_unchanged(before, b.export_state(), "refused arrays (%r)" % bad)
        run_on(cfg, worlds, b, "after the refused arrays")
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("record,evap", MODES, ids=["%s-%s" % c for c in MODES])
def test_non_finite_planes_refused(record, evap):
    """Non-finite pheromone and food values, and in lazy mode pheromone above max_val: ANTS_E_ARG after the window's
    import; importing the window again with clean planes leaves the handle running to parity."""
    from antsrl_b200 import AntsError
    cfg, worlds, b = refusal_handle(record, evap)
    try:
        st = stack_init(cfg, worlds)
        cases = [("phero", v) for v in NON_FINITE] + [("food", v) for v in NON_FINITE]
        if evap == "lazy":
            cases += [("phero", above(MAX)), ("phero", 255.3), ("phero", 1000.0)]
        for key, bad in cases:
            v = np.array(st[key][1:3], copy=True)
            v.reshape(2, -1)[1, 7] = bad
            with pytest.raises(AntsError):
                b.import_state({key: v}, envs=(1, 2))
            b.import_state({key: st[key][1:3]}, envs=(1, 2))
        run_on(cfg, worlds, b, "after the refused planes")
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("record,evap", [("compact8", "lazy"), ("f64", "diffuse")])
def test_bool_activations_map_nan_to_one(record, evap):
    """Bool activations are what numpy's astype(bool) makes of the values: a NaN is True, a deposit of 1.0."""
    import ctypes as C
    from antsrl_b200._cabi import check
    cfg, worlds, b = refusal_handle(record, evap)
    try:
        a = np.zeros((len(worlds), N, P))
        a[:, ::2, 0] = np.nan
        a[:, 1::3, 1] = -0.0
        a[:, 2::3, 1] = 2.0
        check(b.lib, b.lib.ants_activate_all_pheromones(b._h, a.ctypes.data_as(C.c_void_p), 1))
        st = b.export_state()
        assert st["act_bool"]
        assert np.array_equal(st["activation"], a.astype(bool).astype(float))
    finally:
        b.close()
