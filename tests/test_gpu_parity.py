"""GPU parity tests proper: the CUDA path, called through the C ABI, against the oracle on the same seeded
inputs (every step: outputs + full exported state) and against the committed reference-recorded fixtures.
Bar (north_star): integer / index state bit-exact, float state within 1e-5 relative."""
import numpy as np
import pytest

from golden_io import golden_names, load_golden
from parity_util import RTOL, ATOL, assert_close, run_parity, stack_init
from scenarios import GOLDEN_SCENARIOS, make_scenario

pytestmark = pytest.mark.gpu


def _variants(kw, n):
    out = []
    for e in range(n):
        k = dict(kw)
        k["seed"] = kw["seed"] * 100 + e
        out.append(make_scenario(**k))
    return out


@pytest.mark.parametrize("name,kw", GOLDEN_SCENARIOS, ids=[n for n, _ in GOLDEN_SCENARIOS])
@pytest.mark.parametrize("evap_mode", ["dense", "tiles", "lazy", "lazy_compact", "lazy_compact8", "lazy_compact8_flat"])
def test_cuda_matches_oracle_every_step(name, kw, evap_mode, monkeypatch):
    """3 envs per scenario family (different seeds), device-pointer API, taped collision noise; every evaporation
    mode and every cell-record format.  Lazy handles run the block-per-environment kernels (ants_env_fused.cuh);
    "_flat" forces the flat kernels the other modes use onto the 8-byte records as well."""
    kw = dict(kw)
    kw["steps"] = min(kw["steps"], 40)
    record = "f64"
    if evap_mode.endswith("_flat"):
        monkeypatch.setenv("ANTS_NO_FUSED", "1")
        evap_mode = evap_mode[:-5]
    if evap_mode.startswith("lazy_compact"):
        if kw.get("diffuse_factor", 0.0) != 0.0:
            pytest.skip("compact records exist for the lazy (diffusion-free) field only")
        evap_mode, record = "lazy", evap_mode[5:]
    rep = run_parity(_variants(kw, 3), evap_mode=evap_mode, record=record)
    assert rep["kernel_launches"] > 0


@pytest.mark.parametrize("name", golden_names())
def test_cuda_matches_reference_fixture(name):
    """The recorded trajectory of the UNMODIFIED reference (tests/golden) replayed on the GPU, host-buffer API."""
    from antsrl_b200 import BatchedAnts
    cfg, init, tape, rec = load_golden(name)
    batch = BatchedAnts(cfg, 1)
    batch.import_state(stack_init(cfg, [init]))
    obs, ast, st, rew = batch.observe_host()
    assert_close(obs[0], rec["obs0"], "obs0")
    assert_close(ast[0], rec["agent_state0"], "agent_state0")
    assert_close(st[0], rec["state0"], "state0")
    assert_close(rew[0], rec["reward0"], "reward0")
    T = tape["rot"].shape[0]
    for t in range(T):
        rot = None if tape["rot_none"][t] else tape["rot"][t][None].astype(np.int8)
        ph = None if tape["ph_none"][t] else tape["ph"][t][None].astype(np.int8)
        obs, ast, rew, done = batch.step_host(rot, ph)
        assert_close(obs[0], rec["t_obs"][t], "obs t=%d" % t)
        assert_close(ast[0], rec["t_agent_state"][t], "agent_state t=%d" % t)
        assert_close(rew[0], rec["t_reward"][t], "reward t=%d" % t)
        assert done == bool(rec["t_done"][t])
        batch.update_host(tape["noise"][t][None])
        s = batch.export_state(keys=("x", "y", "theta", "holding", "mandibles", "reward_state", "anthill_food",
                                     "rock_centers"))
        pu = rec["t_post_update"][t]
        assert np.array_equal(s["x"][0].astype(np.int64), pu[0].astype(np.int64)), "ant cells x t=%d" % t
        assert np.array_equal(s["y"][0].astype(np.int64), pu[1].astype(np.int64)), "ant cells y t=%d" % t
        assert_close(np.stack([s["x"][0], s["y"][0], s["theta"][0], s["holding"][0]]), pu[:4], "post_update t=%d" % t)
        assert np.array_equal(s["mandibles"][0], pu[4].astype(np.uint8))
        assert np.array_equal(s["reward_state"][0], pu[5].astype(np.uint8))
        assert_close(s["anthill_food"][0], rec["t_anthill_food"][t], "anthill_food t=%d" % t)
        if cfg["n_rocks"]:
            assert_close(s["rock_centers"][0], rec["t_rock_centers"][t], "rock_centers t=%d" % t)
    fin = batch.export_state()
    for k in ("phero", "food", "rw_prev_dist", "rw_holding_prev", "activation", "prev_x", "prev_y"):
        assert_close(fin[k][0], rec["final_" + k], "final " + k)
    for k in ("explored", "walls", "mandibles", "reward_state"):
        assert np.array_equal(fin[k][0], rec["final_" + k]), "final " + k
    assert fin["timestep"] == int(rec["final_timestep"])
    batch.close()


def test_philox_noise_matches_oracle():
    """Throughput mode: in-kernel Philox collision noise, keyed by the global env id."""
    scen = [make_scenario(seed=500 + e, w=48, h=48, n_ants=40, steps=40, n_walls=8) for e in range(4)]
    run_parity(scen, noise_mode="philox", rng_seed=0x1234567890ABCDEF, env_id_base=17)


def test_shard_invariance():
    """E envs on one handle == the same envs split over two handles with env_id_base offsets (multi-GPU
    sharding rule: per-env results do not depend on the partition)."""
    import torch
    from antsrl_b200 import BatchedAnts
    scen = [make_scenario(seed=700 + e, w=48, h=48, n_ants=30, steps=25, n_walls=8) for e in range(6)]
    cfg = scen[0][0]

    def run(sub, base):
        b = BatchedAnts(cfg, len(sub), rng_seed=99, env_id_base=base)
        b.import_state(stack_init(cfg, [i for _, i, _ in sub]))
        b.observe()
        for t in range(25):
            rot = torch.from_numpy(np.stack([s[2]["rot"][t] for s in sub])).cuda()
            ph = torch.from_numpy(np.stack([s[2]["ph"][t] for s in sub])).cuda()
            b.step(rot, ph)
            b.update(None)
        st = b.export_state()
        b.close()
        return st
    whole = run(scen, 0)
    a, c = run(scen[:2], 0), run(scen[2:], 2)
    for k, v in whole.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, np.concatenate([a[k], c[k]])), k


def test_large_batch_properties():
    """Full-size shapes (256x256, 256 ants, 64 envs): size-independent properties instead of the oracle --
    replicated envs stay identical, food is conserved (plane + carried + delivered), explored only grows,
    pheromone stays within [0, max_val] and is zero inside walls after an update."""
    import torch
    from antsrl_b200 import BatchedAnts
    cfg, init, tape = make_scenario(seed=900, w=256, h=256, n_ants=256, steps=30, n_walls=16, n_food=26,
                                    wall_r=(5, 15), food_r=(5, 10))
    E = 64
    for mode in ("dense", "tiles", "lazy", "compact"):
        b = BatchedAnts(cfg, E, evap_mode="lazy" if mode == "compact" else mode,
                        record="compact" if mode == "compact" else "f64")
        b.import_state(stack_init(cfg, [init] * E))
        b.observe()
        total0 = init["food"].sum()
        prev_explored = 0
        for t in range(30):
            rot = torch.from_numpy(np.broadcast_to(tape["rot"][t], (E, 256)).copy()).cuda()
            ph = torch.from_numpy(np.broadcast_to(tape["ph"][t], (E, 256)).copy()).cuda()
            noise = torch.from_numpy(np.broadcast_to(tape["noise"][t], (E, 256)).copy()).cuda()
            b.step(rot, ph)
            b.update(noise)
        st = b.export_state()
        for k, v in st.items():
            if isinstance(v, np.ndarray) and v.size:
                assert np.array_equal(v, np.broadcast_to(v[:1], v.shape)), "replicated envs diverged: " + k
        # no duplicate pickups are possible to rule out (Q1), so conservation is an inequality in general;
        # check the exact identity on env 0 against the oracle-free invariant: nothing negative, nothing lost
        assert (st["food"] >= 0).all() and (st["holding"] >= 0).all()
        assert st["phero"].min() >= 0 and st["phero"].max() <= 255.0
        assert (st["phero"][:, :, st["walls"][0].astype(bool)] == 0).all()
        assert st["explored"].sum() > prev_explored
        assert total0 > 0
        b.close()


ODD_CONFIGS = [
    # radius 1 (9 samples: several ants per lane-slot), one pheromone, no mask, few channels, tiny ant count
    ("r1_p1", dict(seed=31, w=20, h=24, n_ants=7, n_phero=1, steps=25, radius=1, mask=None, fwd_delta=0,
                   channels=["phero0", "food"], none_ph_every=1, n_walls=2, n_food=3, wall_r=(2, 4), food_r=(2, 4))),
    # three pheromones -> 64-byte cell records; activations set through activate_all_pheromones only
    ("p3", dict(seed=32, w=40, h=40, n_ants=33, n_phero=3, steps=30, none_ph_every=1,
                channels=["ants", "phero2", "phero0", "anthill", "walls", "food", "phero1"])),
    # map smaller than the perception reach: samples wrap more than once (slow wrap path)
    ("tiny_map", dict(seed=33, w=9, h=11, n_ants=5, steps=25, n_walls=1, n_food=2, wall_r=(1, 2), food_r=(1, 2))),
    # 11x11 window (121 samples), explore reward, ant count straddling block boundaries
    ("r5_n130", dict(seed=34, w=64, h=48, n_ants=130, steps=20, radius=5, mask=None, fwd_delta=2,
                     channels=["walls", "ants", "food"], reward_kind="explore")),
    # no pheromones at all
    ("p0", dict(seed=35, w=32, h=32, n_ants=20, n_phero=0, steps=20, none_ph_every=1, channels=["ants", "walls", "food", "anthill"])),
    # diffusion on a map of several, partly filled 64x64 stencil tiles (TMA zero fill at every border), with rocks
    ("diffuse_tiles", dict(seed=37, w=130, h=70, n_ants=40, n_rocks=3, steps=20, diffuse_factor=0.03, evap_factor=0.005,
                           n_walls=8, n_food=6)),
    # diffusion with the DEFAULT channel list but windows the row kernel does not serve (radius 4 and 1): the generic
    # kernel must read the f64 planes, not the (empty) record fields
    ("diffuse_r4", dict(seed=38, w=60, h=52, n_ants=40, steps=20, diffuse_factor=0.02, evap_factor=0.01, radius=4,
                        mask=None, fwd_delta=2)),
    ("diffuse_r1", dict(seed=39, w=44, h=40, n_ants=30, steps=20, diffuse_factor=0.03, evap_factor=0.02, radius=1,
                        mask=None, fwd_delta=0)),
    # rocks with a non-default channel list (generic perception path) on a non-square map
    ("rocks_generic", dict(seed=36, w=72, h=56, n_ants=40, n_rocks=5, steps=30,
                           channels=["rocks", "food", "ants", "phero1", "walls"])),
]


@pytest.mark.parametrize("name,kw", ODD_CONFIGS, ids=[n for n, _ in ODD_CONFIGS])
@pytest.mark.parametrize("evap_mode", ["dense", "lazy", "lazy_compact", "lazy_compact8"])
def test_odd_configurations(name, kw, evap_mode):
    record = "f64"
    if evap_mode.startswith("lazy_compact"):
        if kw.get("n_phero", 2) not in (1, 2):
            pytest.skip("compact records hold one or two pheromones")
        if kw.get("diffuse_factor", 0.0) != 0.0:
            pytest.skip("compact records are for the lazy field; diffusion keeps the field in f64 planes")
        evap_mode, record = "lazy", evap_mode[5:]
    rep = run_parity(_variants(kw, 3), evap_mode=evap_mode, record=record)
    assert rep["state_checks"] == kw["steps"]


def test_lazy_timestamp_fold():
    """More updates than the 12-bit timestamp range with float activations: every deposit saturates, so the field holds
    boxed deposits only and the fold passes return at once.  Checks those boxed deposits against the eagerly evaporated
    field (two handles of the CUDA path itself, 4200 updates); the fold's plain-value branches are covered by
    tests/test_gpu_handle_age.py."""
    import torch
    from antsrl_b200 import BatchedAnts
    cfg, init, tape = make_scenario(seed=41, w=32, h=32, n_ants=16, steps=8)
    outs = {}
    for mode in ("tiles", "lazy", "compact", "compact8"):
        b = BatchedAnts(cfg, 2, evap_mode="lazy" if mode.startswith("compact") else mode, rng_seed=5,
                        record=mode if mode.startswith("compact") else "f64")
        b.import_state(stack_init(cfg, [init, init]))
        b.observe()
        for t in range(4200):
            k = t % 8
            if t < 40:
                rot = torch.from_numpy(np.stack([tape["rot"][k]] * 2)).cuda()
                ph = torch.from_numpy(np.stack([tape["ph"][k]] * 2)).cuda()
                b.step(rot, ph)
            b.update(None)
        outs[mode] = b.export_state(keys=("phero", "x"))
        b.close()
    assert np.array_equal(outs["tiles"]["x"], outs["lazy"]["x"])
    assert outs["tiles"]["phero"].max() > 0
    np.testing.assert_allclose(outs["lazy"]["phero"], outs["tiles"]["phero"], rtol=1e-9, atol=0)
    for fmt in ("compact", "compact8"):
        assert np.array_equal(outs["tiles"]["x"], outs[fmt]["x"])
        np.testing.assert_allclose(outs[fmt]["phero"], outs["tiles"]["phero"], rtol=1e-5, atol=0)


@pytest.mark.parametrize("groups", [1, 3], ids=["one_stream", "three_groups"])
@pytest.mark.parametrize("record,n_rocks", [("compact8", 0), ("compact8", 4), ("compact", 0), ("f64", 4)])
def test_rollout_equals_step_update_loop(record, n_rocks, groups, monkeypatch):
    """ants_rollout (device-resident action tapes, C loop; optionally the batch as groups of environments on streams of
    their own) == the same steps issued one by one.  6 envs of 100 ants are 3 blocks of the block-per-env kernel (2 envs
    each), so three groups get one block each; the rollout starts with the anthill sweep of the import pending."""
    import torch
    monkeypatch.setenv("ANTS_ROLLOUT_GROUPS", str(groups))
    from antsrl_b200 import BatchedAnts
    T, E = 12, 6
    scen = [make_scenario(seed=800 + e, w=48, h=48, n_ants=100, n_rocks=n_rocks, steps=T, n_walls=6) for e in range(E)]
    cfg = scen[0][0]
    rot = torch.from_numpy(np.stack([[s[2]["rot"][t] for s in scen] for t in range(T)])).cuda().contiguous()
    ph = torch.from_numpy(np.stack([[s[2]["ph"][t] for s in scen] for t in range(T)])).cuda().contiguous()
    outs = []
    for mode in ("loop", "rollout"):
        b = BatchedAnts(cfg, E, evap_mode="lazy", record=record, rng_seed=3)
        b.import_state(stack_init(cfg, [i for _, i, _ in scen]))
        b.observe()
        if mode == "loop":
            for t in range(T):
                obs, ast, rew, _ = b.step(rot[t], ph[t])
                b.update(None)
        else:
            launches = b.stats()["kernel_launches"]
            obs, ast, rew = b.rollout(rot, ph)
            assert b.stats()["kernel_launches"] - launches >= 2 * groups * T      # every step kernel once per group
        st = b.export_state()
        outs.append((obs.cpu().numpy().copy(), rew.cpu().numpy().copy(), st))
        b.close()
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    for k, v in outs[0][2].items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, outs[1][2][k]), k


@pytest.mark.parametrize("record", ["compact", "compact8", "f64"])
def test_full_size_env_matches_oracle(record):
    """BASELINE configs[3] dimensions (1024x1024 map, 1024 ants, 64 rocks, 7x7x7 obs) for two envs generated by the
    drop-in generator (seeds 1000, 1001), 12 steps with Philox collision noise, compared with the oracle."""
    import torch
    from antsrl_b200 import BatchedAnts
    from antsrl_b200.generator import BatchedEnvironmentGenerator, CirclesGenerator, stack_states
    from oracle.antsrl_oracle import OracleEnv, philox_uniform
    from parity_util import compare_state
    gen = BatchedEnvironmentGenerator(1024, 1024, 1024, 2, 64, CirclesGenerator(320, 5, 10), CirclesGenerator(400, 5, 15),
                                      max_steps=100, seed_base=1000)
    states = gen.generate_states(2, 0)
    cfg = gen.cfg
    oracles = [OracleEnv(cfg, s) for s in states]
    batch = BatchedAnts(cfg, 2, evap_mode="lazy", record=record, rng_seed=11)
    batch.import_state(stack_states(states, "all"))
    act = np.ones((2, 1024, 2)) * 10.0
    batch.activate_all_pheromones(act)
    for o in oracles:
        o.activate_all_pheromones(act[0])
    obs, ast, st, rew = batch.observe()
    ref = [o.observation() for o in oracles]
    assert_close(obs.cpu().numpy(), np.stack([r[0] for r in ref]), "obs0")
    rs = np.random.RandomState(5)
    for t in range(12):
        rot = (rs.randint(0, 3, (2, 1024)) - 1).astype(np.int8)
        ph = rs.randint(0, 3, (2, 1024)).astype(np.int8)
        refs = [o.step(rot[e].astype(np.int64), ph[e].astype(np.int64)) for e, o in enumerate(oracles)]
        obs, ast, rew, done = batch.step(torch.from_numpy(rot).cuda(), torch.from_numpy(ph).cuda())
        assert_close(obs.cpu().numpy(), np.stack([r[0] for r in refs]), "obs %d" % t)
        assert_close(rew.cpu().numpy(), np.stack([r[2] for r in refs]), "reward %d" % t)
        for e, o in enumerate(oracles):
            o.update(philox_uniform(11, e, int(o.s["timestep"]), 1024))
        batch.update(None)
    compare_state(batch.export_state(), oracles, "final (1024x1024)", cfg)
    batch.close()


def _random_config(rng):
    """A random small configuration of the whole path (map, ants, perception window, channels, reward, speeds)."""
    w, h = int(rng.randint(12, 70)), int(rng.randint(12, 70))
    n_rocks = int(rng.choice([0, 0, 3]))
    n_phero = 2
    radius = int(rng.choice([1, 2, 3, 3, 4]))
    s = 2 * radius + 1
    mask = None if rng.rand() < 0.3 else (rng.rand(s, s) < 0.75)
    pool = ["ants", "phero0", "phero1", "anthill", "walls", "food"] + (["rocks"] if n_rocks else [])
    if rng.rand() < 0.5:
        channels = None
    else:
        k = int(rng.randint(2, len(pool) + 1))
        channels = [pool[i] for i in rng.permutation(len(pool))[:k]]
    reward_kind = str(rng.choice(["all", "all", "explore", "food"]))
    kw = dict(seed=int(rng.randint(1, 10 ** 6)), w=w, h=h, n_ants=int(rng.randint(1, 90)), n_rocks=n_rocks,
              n_phero=n_phero, steps=int(rng.randint(8, 22)), n_walls=int(rng.randint(0, 5)), n_food=int(rng.randint(1, 7)),
              wall_r=(1, max(2, min(w, h) // 8)), food_r=(1, max(2, min(w, h) // 8)), radius=radius, mask=mask,
              fwd_delta=float(rng.choice([0, 2, 4])), reward_kind=reward_kind,
              reward_factors=tuple(float(x) for x in rng.choice([0, 1, 2, 5], size=5)),
              reward_threshold=float(rng.choice([0.5, 1.0, 3.0])), max_speed=float(rng.choice([0.6, 1.0, 1.9])),
              max_rot_speed=float(rng.uniform(0.2, 1.2)), carry_speed_reduction=float(rng.choice([0.05, 0.3])),
              backward_speed_reduction=float(rng.choice([0.5, 0.8])), evap_factor=float(rng.choice([0.001, 0.05])),
              float_food=bool(rng.rand() < 0.3), act_float=bool(rng.rand() < 0.7),
              none_rot_every=int(rng.choice([0, 0, 4])), none_ph_every=int(rng.choice([0, 0, 5])))
    if channels is not None:
        kw["channels"] = channels
    return kw


@pytest.mark.parametrize("case", range(24))
def test_random_configurations(case):
    """Seeded fuzz over the configuration space; record format and evaporation mode rotate with the case."""
    rng = np.random.RandomState(9000 + case)
    kw = _random_config(rng)
    mode, record = [("dense", "f64"), ("tiles", "f64"), ("lazy", "f64"), ("lazy", "compact"), ("lazy", "compact8")][case % 5]
    run_parity(_variants(kw, 2), evap_mode=mode, record=record)


@pytest.mark.parametrize("case", range(24, 36))
def test_random_configurations_compact8(case):
    """The bench's cell-record format (8-byte records, lazy field) over twelve more seeded random configurations."""
    kw = _random_config(np.random.RandomState(9000 + case))
    run_parity(_variants(kw, 2), evap_mode="lazy", record="compact8")


def _cmp_outputs(gpu, refs, what):
    obs, ast, rew = [g.cpu().numpy() for g in gpu]
    assert_close(obs, np.stack([r[0] for r in refs]), what + ": obs")
    assert_close(ast, np.stack([r[1] for r in refs]), what + ": agent_state")
    assert_close(rew, np.stack([r[2] for r in refs]), what + ": reward")


@pytest.mark.parametrize("flat", [False, True], ids=["env_kernels", "flat_kernels"])
@pytest.mark.parametrize("record", ["compact", "compact8", "f64"])
@pytest.mark.parametrize("n_rocks", [0, 5])
def test_irregular_call_order(record, n_rocks, flat, monkeypatch):
    """observe / step / update in an order main.py never uses (update before the first step, two steps in a row, two
    updates in a row, a stand-alone observation in between): the per-call bookkeeping the kernels share across calls
    (wall flags written by the move, the double-buffered absorb counter, deposit ownership phases, generation stamps)
    must not depend on strict step/update alternation."""
    import torch
    from antsrl_b200 import BatchedAnts
    from parity_util import compare_state
    from oracle.antsrl_oracle import OracleEnv
    if flat:
        monkeypatch.setenv("ANTS_NO_FUSED", "1")
    scen = [make_scenario(seed=900 + e, w=56, h=48, n_ants=40, n_rocks=n_rocks, steps=16, n_walls=6, n_food=8)
            for e in range(3)]
    cfg = scen[0][0]
    oracles = [OracleEnv(c, i) for c, i, _ in scen]
    b = BatchedAnts(cfg, 3, evap_mode="lazy", record=record)
    b.import_state(stack_init(cfg, [i for _, i, _ in scen]))
    order = "ousussuuosuosusuuussu"
    t = 0
    for k, op in enumerate(order):
        what = "call %d (%s)" % (k, op)
        if op == "o":
            refs = []
            for o in oracles:
                p_, a_, _ = o.observation()
                refs.append((p_, a_, o.s["rewards"].copy()))
            obs, ast, st, rew = b.observe()
            _cmp_outputs((obs, ast, rew), refs, what)
        elif op == "s":
            rot = np.stack([s[2]["rot"][t] for s in scen]).astype(np.int8)
            ph = np.stack([s[2]["ph"][t] for s in scen]).astype(np.int8)
            refs = []
            for e, o in enumerate(oracles):
                p_, a_, r_, _ = o.step(rot[e].astype(np.int64), ph[e].astype(np.int64))
                refs.append((p_, a_, r_.copy()))
            obs, ast, rew, _ = b.step(torch.from_numpy(rot).cuda(), torch.from_numpy(ph).cuda())
            _cmp_outputs((obs, ast, rew), refs, what)
        else:
            noise = np.stack([s[2]["noise"][t] for s in scen])
            for e, o in enumerate(oracles):
                o.update(noise[e])
            b.update(torch.from_numpy(noise).cuda())
            t += 1
        compare_state(b.export_state(), oracles, what, cfg)
    b.close()


@pytest.mark.parametrize("record", ["compact8", "compact"])
def test_reimport_moves_anthill_and_walls(record):
    """A handle is reused for a new episode (main.py:66-79 generates a new map per episode): the second import moves
    the anthill (the disc bit of the cell records), the walls and the rocks; nothing of the first map may survive."""
    import torch
    from antsrl_b200 import BatchedAnts
    from parity_util import compare_state
    from oracle.antsrl_oracle import OracleEnv
    b = None
    for episode, seed0 in enumerate((950, 960)):
        scen = [make_scenario(seed=seed0 + e, w=64, h=64, n_ants=48, n_rocks=4, steps=10, n_walls=5) for e in range(2)]
        cfg = scen[0][0]
        if b is None:
            b = BatchedAnts(cfg, 2, evap_mode="lazy", record=record)
        oracles = [OracleEnv(c, i) for c, i, _ in scen]
        # a COMPLETE state (import leaves missing members untouched): the oracle's own initial state
        b.import_state(stack_init(cfg, [dict(o.s) for o in oracles]))
        refs = []
        for o in oracles:
            p_, a_, _ = o.observation()
            refs.append((p_, a_, o.s["rewards"].copy()))
        obs, ast, st, rew = b.observe()
        _cmp_outputs((obs, ast, rew), refs, "episode %d observation" % episode)
        for t in range(10):
            rot = np.stack([s[2]["rot"][t] for s in scen]).astype(np.int8)
            ph = np.stack([s[2]["ph"][t] for s in scen]).astype(np.int8)
            refs = []
            for e, o in enumerate(oracles):
                p_, a_, r_, _ = o.step(rot[e].astype(np.int64), ph[e].astype(np.int64))
                refs.append((p_, a_, r_.copy()))
            obs, ast, rew, _ = b.step(torch.from_numpy(rot).cuda(), torch.from_numpy(ph).cuda())
            _cmp_outputs((obs, ast, rew), refs, "episode %d step %d" % (episode, t))
            noise = np.stack([s[2]["noise"][t] for s in scen])
            for e, o in enumerate(oracles):
                o.update(noise[e])
            b.update(torch.from_numpy(noise).cuda())
            compare_state(b.export_state(), oracles, "episode %d update %d" % (episode, t), cfg)
    b.close()


def test_crowded_rocks_default_channels():
    """Many rocks on a small map: most ants have several candidate rocks (the multi-rock path of the row-per-lane
    perception kernel), rocks get pushed every step (incremental rock-grid update) and push ants across the seam."""
    kw = dict(seed=970, w=40, h=40, n_ants=64, n_rocks=14, steps=40, n_walls=2, n_food=5)
    for record, mode in (("compact", "lazy"), ("f64", "dense")):
        rep = run_parity(_variants(kw, 3), evap_mode=mode, record=record)
        assert rep["state_checks"] == kw["steps"]


def test_device_action_sampler_matches_oracle_and_sharding():
    """ants_sample_actions: the agents' exploration branch drawn on the device (Philox keyed by global env id, step,
    ant) equals the oracle's mirror, covers the action ranges uniformly and does not depend on the sharding."""
    import torch
    from antsrl_b200 import BatchedAnts
    from oracle.antsrl_oracle import philox_actions
    scen = [make_scenario(seed=990 + e, w=32, h=32, n_ants=96, steps=4) for e in range(4)]
    cfg = scen[0][0]
    whole = BatchedAnts(cfg, 4, evap_mode="lazy", record="compact", env_id_base=10)
    whole.import_state(stack_init(cfg, [i for _, i, _ in scen]))
    halves = [BatchedAnts(cfg, 2, evap_mode="lazy", record="compact", env_id_base=10 + 2 * k) for k in range(2)]
    for k in range(2):
        halves[k].import_state(stack_init(cfg, [i for _, i, _ in scen[2 * k:2 * k + 2]]))
    whole.observe()
    counts = np.zeros((3, 3))
    for t in range(1, 6):
        rot, ph = whole.sample_actions(seed=77)
        rot_h = torch.cat([h.sample_actions(seed=77)[0] for h in halves]).cpu().numpy()
        rot, ph = rot.cpu().numpy(), ph.cpu().numpy()
        assert np.array_equal(rot, rot_h)
        for e in range(4):
            r_ref, p_ref = philox_actions(77, 10 + e, t, 96)
            assert np.array_equal(rot[e], r_ref) and np.array_equal(ph[e], p_ref)
        assert rot.min() == -1 and rot.max() == 1 and ph.min() == 0 and ph.max() == 2
        for a in range(3):
            for b_ in range(3):
                counts[a, b_] += ((rot == a - 1) & (ph == b_)).sum()
        whole.step(torch.from_numpy(rot.astype(np.int8)).cuda(), torch.from_numpy(ph.astype(np.int8)).cuda())
        whole.update(None)
        for h in halves:        # advance the timestep of the halves too (their own random walk)
            r, p = h.sample_actions(seed=77)
            h.step(r, p); h.update(None)
    assert np.abs(counts / counts.sum() - 1 / 9).max() < 0.03
    # five actions: rotation in {-2..2}
    rot5, _ = whole.sample_actions(seed=3, n_rotations=5, n_pheromones=2)
    assert int(rot5.min()) == -2 and int(rot5.max()) == 2
    whole.close()
    for h in halves:
        h.close()


def test_device_replay_memory_ring_buffer():
    """DeviceReplayMemory (agents/replay_memory.py on device tensors): rolling write with wrap-around, the actions
    layout (rotation, pheromone), sampling without replacement -- fed by a random-agent loop that never leaves HBM."""
    import torch
    from antsrl_b200 import BatchedAnts
    from antsrl_b200.replay import DeviceReplayMemory
    scen = [make_scenario(seed=995 + e, w=32, h=32, n_ants=10, steps=4) for e in range(2)]
    cfg = scen[0][0]
    b = BatchedAnts(cfg, 2, evap_mode="lazy", record="compact")
    b.import_state(stack_init(cfg, [i for _, i, _ in scen]))
    mem = DeviceReplayMemory(50, (7, 7, 6), (2,), 2)
    obs, ast, _, _ = b.observe()
    obs, ast = obs.clone(), ast.clone()
    log = []
    for t in range(4):                                   # 4 x 20 entries into 50 slots: wraps once
        rot, ph = b.sample_actions(seed=5)
        new_obs, new_ast, rew, done = b.step(rot, ph)
        mem.extend(obs, ast, (rot, ph), rew, new_obs, new_ast, done)
        log.append((obs.reshape(20, 7, 7, 6).clone(), rot.reshape(-1).clone(), rew.reshape(-1).clone()))
        b.update(None)
        obs, ast = new_obs.clone(), new_ast.clone()
    assert len(mem) == 50 and mem.head == 30
    # slots 0..29 hold entries 50..79 (steps 2 (second half) and 3), slots 30..49 hold entries 30..49 (step 1 tail, step 2 head)
    allobs = torch.cat([l[0] for l in log]); allrot = torch.cat([l[1] for l in log]); allrew = torch.cat([l[2] for l in log])
    assert torch.equal(mem.states[:30], allobs[50:80]) and torch.equal(mem.states[30:], allobs[30:50])
    assert torch.equal(mem.actions[:30, 0], allrot[50:80].to(torch.int64))
    assert torch.allclose(mem.rewards[30:], allrew[30:50].float())
    s = mem.random_access(16)
    assert s[0].shape == (16, 7, 7, 6) and s[2].shape == (16, 2) and s[0].is_cuda
    b.close()


@pytest.mark.parametrize("record", ["compact", "compact8", "f64"])
def test_long_run_crosses_generation_folds(record):
    """300 steps against the oracle: the 7-bit occupancy / exploration generation counters of the compact records fold
    twice (every ~125 steps), the double-buffered commit / absorb counters alternate 300 times."""
    kw = dict(seed=41, w=64, h=56, n_ants=48, n_rocks=3, steps=300, n_walls=5, n_food=8)
    rep = run_parity(_variants(kw, 2), evap_mode="lazy", record=record, state_every=25)
    assert rep["steps"] == 300


def test_parity_with_programmatic_dependent_launch(monkeypatch):
    """Large batches launch the step kernels with programmatic stream serialisation (each kernel may be scheduled while
    its predecessor drains and waits for it with griddepcontrol.wait); the parity batches are small, so force it."""
    monkeypatch.setenv("ANTS_FORCE_PDL", "1")
    for record in ("compact8", "compact"):
        for name in ("rocks", "crowded", "default_small"):
            kw = dict(GOLDEN_SCENARIOS)[name]
            rep = run_parity(_variants(kw, 3), evap_mode="lazy", record=record)
            assert rep["state_checks"] == kw["steps"]


def test_compact8_step_counter_wraps():
    """8-byte records keep 15 bits of a deposit's update index: deposits that have long decayed to zero must not come
    back when the counter wraps (they are cleared every 16384 updates).  33 000 updates against the eagerly evaporated
    field, deposits at the start and again after the wrap."""
    import torch
    from antsrl_b200 import BatchedAnts
    cfg, init, tape = make_scenario(seed=43, w=32, h=32, n_ants=16, steps=8)
    outs = {}
    for mode in ("tiles", "compact8"):
        b = BatchedAnts(cfg, 1, evap_mode="lazy" if mode == "compact8" else mode, rng_seed=5,
                        record=mode if mode == "compact8" else "f64")
        b.import_state(stack_init(cfg, [init]))
        b.observe()
        snaps = []
        for t in range(33000):
            if t < 30 or 32800 <= t < 32830:
                k = t % 8
                b.step(torch.from_numpy(tape["rot"][k][None]).cuda(), torch.from_numpy(tape["ph"][k][None]).cuda())
            if t == 30:                                  # stop depositing (Ants.update emits whatever is activated)
                b.activate_all_pheromones(np.zeros((1, 16, 2)))
            b.update(None)
            if t in (29, 12000, 32799, 32999):
                snaps.append(b.export_state(keys=("phero",))["phero"].copy())
        outs[mode] = snaps
        b.close()
    assert outs["tiles"][0].max() > 0 and outs["tiles"][1].max() == 0 and outs["tiles"][2].max() == 0
    assert outs["tiles"][3].max() > 0
    for a, c in zip(outs["tiles"], outs["compact8"]):
        np.testing.assert_allclose(c, a, rtol=1e-5, atol=0)


def test_generic_perception_kernel_in_diffusion_mode(monkeypatch):
    """ANTS_PERCEIVE_GENERIC routes the default channel list through k_perceive: with DIFFUSE_FACTOR != 0 it must
    read the pheromone planes like k_perceive_rows does (the straight-line record layouts would show zeros)."""
    monkeypatch.setenv("ANTS_PERCEIVE_GENERIC", "1")
    for name in ("diffuse", "rocks", "default_small"):
        kw = dict(dict(GOLDEN_SCENARIOS)[name])
        kw["steps"] = 25
        run_parity(_variants(kw, 2), evap_mode="dense")
    kw = dict(dict(GOLDEN_SCENARIOS)["default_small"], steps=25)
    run_parity(_variants(kw, 2), evap_mode="lazy", record="compact8")


def test_lazy_mode_rejects_slow_evaporation():
    """A max_val deposit that does not decay below 0.01 within the 16384-entry table cannot be boxed: ants_create
    refuses lazy evaporation for such factors instead of silently zeroing the field at age 16384; the eager modes
    take them."""
    from antsrl_b200 import BatchedAnts, AntsError
    cfg, init, tape = make_scenario(seed=45, w=32, h=32, n_ants=8, steps=4, evap_factor=0.0005)
    with pytest.raises(AntsError, match="evap_factor"):
        BatchedAnts(cfg, 1, evap_mode="lazy", record="compact8")
    with pytest.raises(AntsError, match="evap_factor"):
        BatchedAnts(cfg, 1, evap_mode="lazy")
    run_parity([(cfg, init, tape)], evap_mode="tiles")


def test_partial_import_keeps_scalars():
    """Patching positions mid-episode must not rewind the timestep (done flag, Philox counter), flip the activation
    dtype (deposit strength 256 vs 1) or re-alias the reward."""
    import torch
    from antsrl_b200 import BatchedAnts
    cfg, init, tape = make_scenario(seed=46, w=32, h=32, n_ants=12, steps=6)
    b = BatchedAnts(cfg, 1, evap_mode="lazy", record="compact8")
    b.import_state(stack_init(cfg, [init]))
    b.observe()
    for t in range(3):
        b.step(torch.from_numpy(tape["rot"][t][None]).cuda(), torch.from_numpy(tape["ph"][t][None]).cuda())
        b.update(None)
    before = b.export_state()
    b.import_state({"x": before["x"], "y": before["y"]})
    after = b.export_state()
    assert after["timestep"] == before["timestep"] == 4
    assert after["act_bool"] == before["act_bool"] and after["rw_alias"] == before["rw_alias"] is False
    for k in ("holding", "phero", "food", "explored", "theta"):
        assert np.array_equal(before[k], after[k]), k
    b.close()


@pytest.mark.parametrize("groups", [1, 4], ids=["one_stream", "four_groups"])
@pytest.mark.parametrize("record,n_rocks,n_ants,n_envs", [("compact8", 6, 300, 3), ("compact8", 0, 50, 7), ("compact", 4, 520, 2),
                                                          ("f64", 3, 1024, 2), ("compact8", 2, 1100, 2)])
def test_rollout_matches_oracle(record, n_rocks, n_ants, n_envs, groups, monkeypatch):
    """ants_rollout (update_k and the move of step_{k+1} in ONE launch of the block-per-environment kernel; 1 or 2
    ants per thread, several envs per block for small N; 1100 ants per env falls back to the flat kernels) against the
    oracle: last observation / reward and the full final state after 30 steps, Philox noise, crowded hill (shared
    cells: the last-writer scatters) and food near it."""
    import torch
    from antsrl_b200 import BatchedAnts
    from oracle.antsrl_oracle import OracleEnv, philox_uniform
    from parity_util import compare_state
    monkeypatch.setenv("ANTS_ROLLOUT_GROUPS", str(groups))
    T = 30
    scen = [make_scenario(seed=1200 + e, w=72, h=64, n_ants=n_ants, n_rocks=n_rocks, steps=T, n_walls=6, n_food=14)
            for e in range(n_envs)]
    cfg = scen[0][0]
    oracles = [OracleEnv(c, i) for c, i, _ in scen]
    b = BatchedAnts(cfg, n_envs, evap_mode="lazy", record=record, rng_seed=21, env_id_base=5)
    b.import_state(stack_init(cfg, [i for _, i, _ in scen]))
    b.observe()
    for o in oracles:
        o.observation()
    rot = torch.from_numpy(np.stack([[s[2]["rot"][t] for s in scen] for t in range(T)])).cuda().contiguous()
    ph = torch.from_numpy(np.stack([[s[2]["ph"][t] for s in scen] for t in range(T)])).cuda().contiguous()
    obs, ast, rew = b.rollout(rot, ph)
    refs = []
    for e, o in enumerate(oracles):
        for t in range(T):
            r = o.step(scen[e][2]["rot"][t].astype(np.int64), scen[e][2]["ph"][t].astype(np.int64))
            o.update(philox_uniform(21, 5 + e, int(o.s["timestep"]), n_ants))
        refs.append(r)
    _cmp_outputs((obs, ast, rew), refs, "last step of the rollout")
    compare_state(b.export_state(), oracles, "after the rollout", cfg)
    b.close()


@pytest.mark.parametrize("record,n_rocks", [("compact8", 3), ("f64", 0)])
def test_windowed_import_resets_some_environments(record, n_rocks):
    """ants_import_env_state: a batch uploaded in two slices equals the batch uploaded at once, and a new episode for
    ONE environment in the middle of the others' (main.py:66-79 generates a new map per episode) leaves its neighbours
    untouched: everything is compared with the oracle after every step."""
    import torch
    from antsrl_b200 import BatchedAnts
    from parity_util import compare_state
    from oracle.antsrl_oracle import OracleEnv
    T = 24
    scen = [make_scenario(seed=1400 + e, w=56, h=48, n_ants=40, n_rocks=n_rocks, steps=T, n_walls=5, n_food=8) for e in range(5)]
    cfg = scen[0][0]
    oracles = [OracleEnv(c, i) for c, i, _ in scen[:4]]
    b = BatchedAnts(cfg, 4, evap_mode="lazy", record=record)
    b.import_state(stack_init(cfg, [i for _, i, _ in scen[:3]]), envs=(0, 3))      # two slices
    b.import_state(stack_init(cfg, [scen[3][1]]), envs=(3, 1))
    b.observe()
    for o in oracles:
        o.observation()
    src = [0, 1, 2, 3]                       # which scenario's tape drives env e
    t_env = [0, 0, 0, 0]
    for t in range(T):
        if t == 9:
            # env 2 starts a new episode on scenario 4's map; the timestep stays the batch's (lockstep)
            fresh = OracleEnv(cfg, scen[4][1])
            fresh.s["timestep"] = int(oracles[0].s["timestep"])
            st = stack_init(cfg, [dict(fresh.s)])
            st.pop("timestep", None); st.pop("rw_alias", None); st.pop("act_bool", None)
            b.import_state(st, envs=(2, 1))
            fresh.s["rw_alias"] = oracles[0].s["rw_alias"]       # batch-wide flag (the reward no longer aliases holding)
            fresh.s["rw_holding_prev"] = fresh.s["holding"].copy()
            oracles[2] = fresh
            src[2], t_env[2] = 4, 0
        rot = np.stack([scen[src[e]][2]["rot"][t_env[e]] for e in range(4)]).astype(np.int8)
        ph = np.stack([scen[src[e]][2]["ph"][t_env[e]] for e in range(4)]).astype(np.int8)
        refs = []
        for e, o in enumerate(oracles):
            p_, a_, r_, _ = o.step(rot[e].astype(np.int64), ph[e].astype(np.int64))
            refs.append((p_, a_, r_.copy()))
        obs, ast, rew, _ = b.step(torch.from_numpy(rot).cuda(), torch.from_numpy(ph).cuda())
        _cmp_outputs((obs, ast, rew), refs, "step %d" % t)
        noise = np.stack([scen[src[e]][2]["noise"][t_env[e]] for e in range(4)])
        for e, o in enumerate(oracles):
            o.update(noise[e])
        b.update(torch.from_numpy(noise).cuda())
        compare_state(b.export_state(), oracles, "after update %d" % t, cfg)
        for e in range(4):
            t_env[e] += 1
    b.close()


def test_grouped_rollout_crosses_generation_folds(monkeypatch):
    """260 steps of ants_rollout with the batch split into groups on their own streams: the 7-bit generation counters of
    the compact records fold twice on the way and the lazy field's update counter once (whole-batch passes that must
    join the groups first and fork them again).  12 envs of 48 ants are 3 blocks of the block-per-env kernel (5 envs
    each, the last one partial), one per group."""
    import torch
    from antsrl_b200 import BatchedAnts
    from oracle.antsrl_oracle import OracleEnv, philox_uniform
    from parity_util import compare_state
    G = 3
    monkeypatch.setenv("ANTS_ROLLOUT_GROUPS", str(G))
    T, E, N = 260, 12, 48
    scen = [make_scenario(seed=1700 + e, w=64, h=56, n_ants=N, n_rocks=3, steps=T, n_walls=5, n_food=8) for e in range(E)]
    cfg = scen[0][0]
    oracles = [OracleEnv(c, i) for c, i, _ in scen]
    b = BatchedAnts(cfg, E, evap_mode="lazy", record="compact8", rng_seed=31)
    b.import_state(stack_init(cfg, [i for _, i, _ in scen]))
    b.observe()
    for o in oracles:
        o.observation()
    rot = torch.from_numpy(np.stack([[s[2]["rot"][t] for s in scen] for t in range(T)])).cuda().contiguous()
    ph = torch.from_numpy(np.stack([[s[2]["ph"][t] for s in scen] for t in range(T)])).cuda().contiguous()
    launches = b.stats()["kernel_launches"]
    obs, ast, rew = b.rollout(rot[:100], ph[:100])           # two calls: the second one starts with move_done cleared
    obs, ast, rew = b.rollout(rot[100:], ph[100:])
    launches = b.stats()["kernel_launches"] - launches
    refs = []
    for e, o in enumerate(oracles):
        for t in range(T):
            r = o.step(scen[e][2]["rot"][t].astype(np.int64), scen[e][2]["ph"][t].astype(np.int64))
            o.update(philox_uniform(31, e, int(o.s["timestep"]), N))
        refs.append(r)
    _cmp_outputs((obs, ast, rew), refs, "last step of the grouped rollout")
    compare_state(b.export_state(), oracles, "after the grouped rollout", cfg)
    assert launches >= 2 * G * T                               # every step kernel once per group
    b.close()


@pytest.mark.parametrize("record", ["compact8", "compact", "f64"])
def test_row_kernel_5x5_window_with_rocks(record):
    """The 5x5 window of the row-per-lane kernel (radius 2, S = 5) with rocks and the default channel list: the rock
    channel of an ant a rock can reach is evaluated by the whole warp, 25 samples in one pass, and handed back to the
    ant's five row lanes (ants_perceive_rows.cuh, rock_rows); RL_api.py:132-135."""
    for seed in (501, 502):
        scen = [make_scenario(seed=seed + 10 * e, w=48, h=40, n_ants=70, n_rocks=5, steps=14, radius=2, mask=None, fwd_delta=2)
                for e in range(3)]
        report = run_parity(scen, evap_mode="lazy", record=record)
        assert report["state_checks"] == 14
