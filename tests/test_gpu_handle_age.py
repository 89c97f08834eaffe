"""Parity across the counters that measure a handle's age rather than its episode's.

A handle reused across episodes (main.py:66-79, any training loop) keeps counting updates and observations in host
counters of ants_abi.cu, and each counter has a fold or reset pass that runs only when it is about to wrap:

* lazy_now, the small write timestamp of plain pheromone values: k_lazy_fold re-bases them every 254 updates (8- and
  16-byte records) or 4094 updates (f64 records);
* lazy_abs, the 22-bit update index of boxed saturated deposits: k_lazy_fold unboxes them into plain values every
  2^22 - 3 updates (f64, 16-byte records), or clears expired ones every 16 384 updates (8-byte records);
* obs_gen / occ_gen, the 16-bit exploration and occupancy stamps of f64 records: k_meta_renormalize folds them every
  65 532 observations;
* owner_phase, the deposit ownership phase of the flat kernels: a memset every 0xFFFE phases (two per iteration).

An import keeps lazy_now and lazy_abs; a whole-batch import with `explored` restarts obs_gen / occ_gen and every import
restarts owner_phase.  The tests advance a handle cheaply to just before a wrap (ants_rollout, no Python per step),
then run it against the oracle in lockstep through the wrap.  `Clock` mirrors the host counters from the calls the
test makes; each test checks that the predicted wraps fell inside its lockstep window and that the launch counts of
the window agree (k_lazy_fold is the `evaporate` family of a lazy handle; `misc` counts k_meta_renormalize only).
"""
import copy

import numpy as np
import pytest

from oracle.antsrl_oracle import OracleEnv, philox_uniform
from parity_util import assert_close, compare_state, stack_init
from scenarios import make_scenario

pytestmark = pytest.mark.gpu

CUT = 0.01                    # pheromone.py:45: values below it are zeroed after evaporation
UNBOX_AT = (1 << 22) - 3      # lazy_abs that makes the next update unbox (f64 and 16-byte records)
CLEAR8 = 0x3FFF               # 8-byte records: expired boxed deposits are cleared when lazy_abs & CLEAR8 == CLEAR8
LEAD = 300                    # lockstep iterations before the wrap a test is after


def _restarts(v, lim, n):
    """n calls of a counter that restarts (reset to 0, then incremented) at the call finding it >= lim, as the
    counters of ants_abi.cu do.  -> (value after the n calls, offsets of the restarting calls)"""
    hits, i = [], 0
    while True:
        k = max(lim - v, 0)
        if i + k >= n:
            return v + (n - i), hits
        i += k
        hits.append(i)
        v, i = 1, i + 1


class Clock:
    """The host counters of one handle, advanced for every call the test makes on it.  `steps` counts iterations
    (step + update) since the handle was created; `events` lists (kind, iteration) of every fold or reset."""

    def __init__(self, record, lazy, flat):
        self.record, self.lazy, self.flat = record, lazy, flat
        self.ts_lim = (0xFFF if record == "f64" else 0xFF) - 1          # fold when lazy_now >= ts_mask - 1
        self.gen_lim = (0xFFFF if record == "f64" else 0x7F) - 3         # maybe_fold_generations (obs_gen == occ_gen)
        self.now = self.abs = self.gen = self.phase = 0
        self.steps = 0
        self.events = []

    def _gen(self, n):
        self.gen, hits = _restarts(self.gen, self.gen_lim, n)
        return hits

    def _owner(self, n):
        if not self.flat:
            return []
        self.phase, hits = _restarts(self.phase, 0xFFFE, n)
        return hits

    def _lazy(self, n):
        if not self.lazy:
            return
        rec8, i = self.record == "compact8", 0
        while True:
            to_now = max(self.ts_lim - self.now, 0)
            to_box = ((CLEAR8 - self.abs) & CLEAR8) if rec8 else max(UNBOX_AT - self.abs, 0)
            k = min(to_now, to_box)
            if i + k >= n:
                self.now += n - i
                self.abs += n - i
                return
            i += k
            self.now += k
            self.abs += k
            unbox = k == to_box
            self.events.append(("unbox" if unbox else "fold", self.steps + i))
            self.now = 1
            self.abs = 1 if unbox and not rec8 else self.abs + 1
            i += 1

    def import_whole(self):
        """A whole-batch import with `explored`: the generation stamps and the owner phase restart."""
        self.gen = self.phase = 0

    def observe(self):
        self.events += [("gen", self.steps) for _ in self._gen(1)]

    def advance(self, n):
        """n iterations of [step; update]."""
        self.events += [("gen", self.steps + j) for j in self._gen(n)]
        self.events += [("owner", self.steps + j // 2) for j in self._owner(2 * n)]
        self._lazy(n)
        self.steps += n

    def predict(self, n):
        """Events of the next n iterations, as (kind, iteration within the window)."""
        probe = copy.deepcopy(self)
        probe.events = []
        probe.advance(n)
        return sorted((k, i - self.steps) for k, i in probe.events)

    def next_event(self, kind, horizon):
        return min(i for k, i in self.predict(horizon) if k == kind) + self.steps


def make_handle(cfg, record, evap_mode, monkeypatch, env=()):
    from antsrl_b200 import BatchedAnts
    for k, v in env:
        monkeypatch.setenv(k, v)
    b = BatchedAnts(cfg, 1, evap_mode=evap_mode, record=record, rng_seed=9)
    flat = evap_mode != "lazy" or cfg["diffuse_factor"] != 0.0 or dict(env).get("ANTS_NO_FUSED") == "1"
    return b, Clock(record, evap_mode == "lazy", flat)


def new_episode(b, clock, cfg, init):
    """Import a complete state (the oracle's initial state, timestep 1) into the reused handle and make the main.py
    observation; -> the oracles."""
    oracles = [OracleEnv(cfg, init)]
    b.import_state(stack_init(cfg, [dict(o.s) for o in oracles]))
    clock.import_whole()
    obs, ast, _, rew = b.observe()
    clock.observe()
    refs = []
    for o in oracles:
        p_, a_, _ = o.observation()
        refs.append((p_, a_, o.s["rewards"].copy()))
    _cmp_outputs((obs, ast, rew), refs, "observation of the new episode", None, cfg)
    return oracles


def oracles_from_handle(b, cfg):
    """Continue the handle's episode on the oracle: one oracle per env, started from the exported state."""
    st = b.export_state()
    return [OracleEnv(cfg, {k: (v[e] if isinstance(v, np.ndarray) else v) for k, v in st.items()}) for e in range(b.E)]


def fast_forward(b, clock, n, chunk=1 << 20):
    """Advance the handle by n iterations with no pheromone deposits (float zero activations: nothing plain is
    stored and no saturated deposit either), None actions and Philox noise, in ants_rollout chunks."""
    b.activate_all_pheromones(np.zeros((b.E, b.N, b.P)))
    done = 0
    while done < n:
        k = min(chunk, n - done)
        b.rollout(None, None, n_steps=k)
        done += k
    b.synchronize()
    clock.advance(n)


def _exempt(gpu, ref, cut):
    """gpu with the entries that land on the other side of the reference's < 0.01 cut set to the oracle's value: one
    side is 0 and the other lies within 1e-6 relative of the cut (f32 plain values of the compact records)."""
    gpu = np.array(gpu, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    if cut is None:
        return gpu, 0
    other = np.where(gpu == 0.0, ref, gpu)
    m = ((gpu == 0.0) != (ref == 0.0)) & (np.abs(other - cut) <= 1e-6 * cut)
    gpu[m] = ref[m]
    return gpu, int(m.sum())


def _cmp_outputs(gpu, refs, what, cut, cfg):
    obs, ast, rew = [g.cpu().numpy() if hasattr(g, "cpu") else np.asarray(g) for g in gpu]
    ref_obs = np.stack([r[0] for r in refs])
    obs, n = _exempt(obs, ref_obs, None if cut is None else cut / cfg["phero_max_val"])
    assert_close(obs, ref_obs, what + ": obs")
    assert_close(ast, np.stack([r[1] for r in refs]), what + ": agent_state")
    assert_close(rew, np.stack([r[2] for r in refs]), what + ": reward")
    return n


def _cmp_state(b, oracles, what, cut, cfg):
    st = b.export_state()
    st["phero"], n = _exempt(st["phero"], np.stack([o.s["phero"] for o in oracles]), cut)
    compare_state(st, oracles, what, cfg)
    return n


def lockstep(b, clock, oracles, cfg, tape, n, every=25, cut=None, rollout=False, use_ph=True):
    """n iterations on the handle and the oracles from the tape's first row: taped actions (pheromone actions only
    with use_ph), taped collision noise -- or with `rollout` ants_rollout chunks and Philox noise.  Observation,
    agent state and reward are compared after every step (rollout: at the end of every chunk); the full state every
    `every` iterations and at every iteration within 3 of a predicted wrap (rollout: the chunks end there).
    -> (predicted events of the window, launches per kernel family in the window, exempted entries)"""
    import torch
    events = clock.predict(n)
    checks = set(range(every - 1, n, every)) | {n - 1}
    checks |= {i + d for _, i in events for d in range(-3, 4) if 0 <= i + d < n}
    dev = b.device
    E = b.E
    exempted = 0
    b.reset_kernel_ms()
    if rollout:
        ends = sorted(checks)
        starts = [0] + [e + 1 for e in ends[:-1]]
        for t0, t1 in zip(starts, ends):
            rot = torch.from_numpy(np.ascontiguousarray(tape["rot"][t0:t1 + 1, None])).to(dev)
            ph = torch.from_numpy(np.ascontiguousarray(tape["ph"][t0:t1 + 1, None])).to(dev) if use_ph else None
            obs, ast, rew = b.rollout(rot, ph)
            for t in range(t0, t1 + 1):
                refs = []
                for e, o in enumerate(oracles):
                    p_, a_, r_, _ = o.step(tape["rot"][t].astype(np.int64), tape["ph"][t].astype(np.int64) if use_ph else None)
                    refs.append((p_, a_, r_.copy()))
                    o.update(philox_uniform(9, e, int(o.s["timestep"]), cfg["n_ants"]))
            what = "rollout to iteration %d" % t1
            exempted += _cmp_outputs((obs, ast, rew), refs, what, cut, cfg)
            exempted += _cmp_state(b, oracles, what, cut, cfg)
    else:
        for t in range(n):
            rot = np.broadcast_to(tape["rot"][t], (E, b.N)).astype(np.int8)
            ph = np.broadcast_to(tape["ph"][t], (E, b.N)).astype(np.int8)
            refs = []
            for e, o in enumerate(oracles):
                p_, a_, r_, d_ = o.step(rot[e].astype(np.int64), ph[e].astype(np.int64) if use_ph else None)
                refs.append((p_, a_, r_.copy(), d_))
            obs, ast, rew, done = b.step(torch.from_numpy(rot).to(dev), torch.from_numpy(ph).to(dev) if use_ph else None)
            exempted += _cmp_outputs((obs, ast, rew), refs, "iteration %d" % t, cut, cfg)
            assert done == refs[0][3], "done at iteration %d" % t
            noise = np.broadcast_to(tape["noise"][t], (E, b.N))
            for e, o in enumerate(oracles):
                o.update(noise[e])
            b.update(torch.from_numpy(np.ascontiguousarray(noise)).to(dev))
            if t in checks:
                exempted += _cmp_state(b, oracles, "after update %d" % t, cut, cfg)
    clock.advance(n)
    launches = {k: v[1] for k, v in b.kernel_ms().items()}
    return events, launches, exempted


def _inside(events, kind, n, count=1):
    """The window's wraps of `kind`: at least `count` of them, each with room for the checks around it."""
    at = [i for k, i in events if k == kind]
    assert len(at) >= count, "expected %d %s wraps in the window, predicted %r" % (count, kind, events)
    assert all(3 <= i < n - 3 for i in at), "%s wraps %r too close to the window's edges" % (kind, at)
    return at


# ---------------------------------------------------------------------------------------- 1. plain values, lazy_now
PLAIN_CASES = [
    ("f64_p2", "f64", 2, False, ()),
    ("f64_p2_flat", "f64", 2, False, (("ANTS_NO_FUSED", "1"),)),
    ("f64_p3", "f64", 3, False, ()),
    ("f64_p3_flat", "f64", 3, False, (("ANTS_NO_FUSED", "1"),)),
    ("compact", "compact", 2, False, ()),
    ("compact_flat", "compact", 2, False, (("ANTS_NO_FUSED", "1"),)),
    ("compact_generic", "compact", 2, False, (("ANTS_PERCEIVE_GENERIC", "1"),)),
    ("compact_rollout", "compact", 2, True, ()),
    ("compact8", "compact8", 2, False, ()),
    ("compact8_flat", "compact8", 2, False, (("ANTS_NO_FUSED", "1"),)),
    ("compact8_rollout", "compact8", 2, True, ()),
]


@pytest.mark.parametrize("name,record,P,rollout,env", PLAIN_CASES, ids=[c[0] for c in PLAIN_CASES])
def test_plain_values_across_timestamp_folds(name, record, P, rollout, env, monkeypatch):
    """Plain (non-saturated) pheromone values across two or more folds of the small write timestamp, from the first
    step against the oracle.  Two pheromones: bool activations (the pheromone action deposits 1.0) with walls on the
    map; three: float activations of 3.7 and no pheromone actions.  The 8-byte records also hold non-integer food (its
    escape sets the plain-value flag as well)."""
    n = 8300 if record == "f64" else 600
    cfg, init, tape = make_scenario(seed=2100 + P, w=24, h=20, n_ants=8, n_phero=P, steps=n, n_walls=3, n_food=3,
                                    act_float=P != 2, float_food=record == "compact8")
    b, clock = make_handle(cfg, record, "lazy", monkeypatch, env)
    oracles = [OracleEnv(cfg, init)]
    b.import_state(stack_init(cfg, [init]))
    clock.import_whole()
    if P != 2:
        act = np.full((1, 8, P), 3.7)
        b.activate_all_pheromones(act)
        oracles[0].activate_all_pheromones(act[0])
    obs, ast, _, rew = b.observe()
    clock.observe()
    p_, a_, _ = oracles[0].observation()
    _cmp_outputs((obs, ast, rew), [(p_, a_, oracles[0].s["rewards"].copy())], "observation", None, cfg)
    cut = None if record == "f64" else CUT
    events, launches, exempted = lockstep(b, clock, oracles, cfg, tape, n, cut=cut, rollout=rollout, use_ph=P == 2)
    b.close()
    folds = _inside(events, "fold", n, count=2)
    assert launches["evaporate"] == len([e for e in events if e[0] in ("fold", "unbox")]), (launches, events)
    field = oracles[0].s["phero"]
    assert ((field > 0) & (field < cfg["phero_max_val"])).any(), "the oracle's field holds no plain value"
    print("%s: folds at %r, %d entries exempted at the cut" % (name, folds, exempted))


# ---------------------------------------------------------- 2. 16-bit generation stamps and the owner phase reset
GEN_MODES = [
    ("dense", "dense", 0.0, ()),
    ("tiles", "tiles", 0.0, ()),
    ("lazy", "lazy", 0.0, ()),
    ("lazy_flat", "lazy", 0.0, (("ANTS_NO_FUSED", "1"),)),
    ("diffusion", "dense", 0.02, ()),
    ("dense_pdl", "dense", 0.0, (("ANTS_FORCE_PDL", "1"),)),
]


@pytest.mark.parametrize("reward", ["all", "explore"])
@pytest.mark.parametrize("name,evap_mode,diffuse,env", GEN_MODES, ids=[m[0] for m in GEN_MODES])
def test_f64_generation_folds_and_owner_phase_reset(name, evap_mode, diffuse, env, reward, monkeypatch):
    """f64 records stamp exploration and occupancy with 16-bit generations, folded every 65 532 observations; the
    flat kernels' ownership phase restarts every 32 767 iterations.  Both restart at a whole-batch import, so a
    single long episode crosses them: the handle runs to 300 iterations before each wrap, the oracle continues the
    episode from the exported state, and 600 iterations run in lockstep.  The default channel list shows occupancy
    (`ants`), and both rewards read exploration: a stale or wrongly folded stamp changes the observation or reward."""
    n = 600
    cfg, init, tape = make_scenario(seed=2200, w=24, h=20, n_ants=8, steps=n, n_walls=3, n_food=3, reward_kind=reward,
                                    diffuse_factor=diffuse, max_time=1 << 30)
    b, clock = make_handle(cfg, "f64", evap_mode, monkeypatch, env)
    b.import_state(stack_init(cfg, [init]))
    clock.import_whole()
    b.observe()
    clock.observe()
    windows = (["owner"] if clock.flat else []) + ["gen"]
    for kind in windows:
        fast_forward(b, clock, clock.next_event(kind, 70000) - LEAD - clock.steps)
        oracles = oracles_from_handle(b, cfg)
        events, launches, _ = lockstep(b, clock, oracles, cfg, tape, n)
        at = _inside(events, kind, n)
        assert at[0] == LEAD
        assert launches["misc"] == len([e for e in events if e[0] == "gen"]), (launches, events)
        print("%s/%s: %s window, events %r, clock at %d iterations" % (name, reward, kind, events, clock.steps))
    b.close()


# ------------------------------------------------------------------------------------- 3. the unboxing fold
UNBOX_CASES = [
    ("f64", "f64", ()),
    ("f64_generic", "f64", (("ANTS_PERCEIVE_GENERIC", "1"),)),
    ("compact", "compact", ()),
    ("compact_generic", "compact", (("ANTS_PERCEIVE_GENERIC", "1"),)),
    ("compact8", "compact8", ()),
]


@pytest.mark.parametrize("name,record,env", UNBOX_CASES, ids=[c[0] for c in UNBOX_CASES])
def test_unboxing_fold(name, record, env, monkeypatch):
    """Float activations only (every deposit saturates and is boxed, so no plain value exists before the fold).  The
    handle runs to 300 updates before lazy_abs makes k_lazy_fold unbox (2^22 - 3 updates; 8-byte records: the clear of
    expired deposits every 16 384), a new episode with taped pheromone actions puts live deposits into the field, and
    the lockstep runs through the unbox and past the next fold of the small timestamp (8-byte records: through two
    clears).  The unboxed deposits must keep showing and keep decaying as the oracle's field does."""
    rec8 = record == "compact8"
    n = {"f64": LEAD + 4200, "compact": LEAD + 300, "compact8": LEAD + 16384 + 300}[record]
    cfg, init, tape = make_scenario(seed=2300, w=24, h=20, n_ants=8, steps=n, n_walls=3, n_food=3, max_time=1 << 30)
    b, clock = make_handle(cfg, record, "lazy", monkeypatch, env)
    b.import_state(stack_init(cfg, [init]))
    clock.import_whole()
    fast_forward(b, clock, clock.next_event("unbox", 1 << 23) - LEAD - clock.steps)
    oracles = new_episode(b, clock, cfg, init)
    events, launches, exempted = lockstep(b, clock, oracles, cfg, tape, n, cut=None if record == "f64" else CUT)
    b.close()
    unboxes = _inside(events, "unbox", n, count=2 if rec8 else 1)
    assert unboxes[0] == LEAD
    if not rec8:
        assert any(k == "fold" and i > unboxes[0] for k, i in events), events
    assert launches["evaporate"] == len([e for e in events if e[0] in ("fold", "unbox")]), (launches, events)
    print("%s: events %r, %d entries exempted at the cut" % (name, events, exempted))
