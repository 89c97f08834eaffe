"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on the seeded
scenarios of tests/scenarios.py.  Run in the build container only:

    python tests/golden/make_golden.py            # writes tests/golden/<name>.npz

Driver loop = main.py:88-138: one extra observation(), then T x [step(actions_t); env.update()].
The wall-collision draws of walls.py:28 are taped (ref_harness.py) so the trajectory is a pure function of
(initial state, action tape, noise tape).  Everything recorded is reference output; nothing here is computed
by the oracle or the CUDA path.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import ref_harness  # noqa: E402
from scenarios import GOLDEN_SCENARIOS, make_scenario  # noqa: E402

PER_STEP_ANT_KEYS = ["x", "y", "theta", "prev_x", "prev_y", "holding", "mandibles", "reward_state", "activation"]


def cfg_to_json(cfg):
    c = dict(cfg)
    c["mask"] = None if cfg["mask"] is None else np.asarray(cfg["mask"]).astype(int).tolist()
    return json.dumps(c)


def run_reference(cfg, init, tape):
    ref = ref_harness.load_reference()
    ref_harness.set_diffuse(ref, cfg["diffuse_factor"], cfg["evap_factor"])
    env, api, objs = ref_harness.build_env(ref, cfg, init)
    if not init.get("act_bool", True):
        objs["ants"].activate_all_pheromones(np.asarray(init["activation"], dtype=float))
    rec = {}
    obs0, agent_state0, state0 = api.observation()
    rec["obs0"] = obs0; rec["agent_state0"] = agent_state0; rec["state0"] = state0
    rec["reward0"] = np.asarray(api.reward.rewards, dtype=float).copy()
    T = tape["rot"].shape[0]
    per = {"obs": [], "agent_state": [], "reward": [], "done": [], "post_step": [], "post_update": [],
           "phero_sum": [], "food_sum": [], "explored_count": [], "anthill_food": [], "rock_centers": []}
    for t in range(T):
        rot = None if tape["rot_none"][t] else tape["rot"][t].astype(np.int64)
        ph = None if tape["ph_none"][t] else tape["ph"][t].astype(np.int64)
        obs, agent_state, reward, done = api.step(rot, ph)
        per["obs"].append(obs); per["agent_state"].append(agent_state)
        per["reward"].append(np.asarray(reward, dtype=float).copy()); per["done"].append(bool(done))
        st = ref_harness.export_state(env, api, objs)
        per["post_step"].append(np.stack([st["x"], st["y"], st["theta"], st["holding"],
                                          st["mandibles"].astype(float), st["reward_state"].astype(float)]))
        ref_harness.run_update(ref, env, tape["noise"][t])
        st = ref_harness.export_state(env, api, objs)
        per["post_update"].append(np.stack([st["x"], st["y"], st["theta"], st["holding"],
                                            st["mandibles"].astype(float), st["reward_state"].astype(float)]))
        per["phero_sum"].append(st["phero"].sum(axis=(1, 2)))
        per["food_sum"].append(st["food"].sum())
        per["explored_count"].append(int(st["explored"].sum()))
        per["anthill_food"].append(float(st["anthill_food"]))
        per["rock_centers"].append(st["rock_centers"].copy())
    final = ref_harness.export_state(env, api, objs)
    for k, v in per.items():
        rec["t_" + k] = np.array(v)
    for k, v in final.items():
        rec["final_" + k] = np.asarray(v)
    rec["wall_hits"] = np.int64(ref.walls_proxy.hits)
    ref.walls_proxy.hits = 0
    return rec


def save_npz(path, arrays):
    """np.savez with bzip2-compressed members (np.load reads them): the per-step observations of a scenario compress
    to well under 1 MB this way, about a third smaller than with np.savez_compressed."""
    import zipfile
    with zipfile.ZipFile(path, "w", zipfile.ZIP_BZIP2, compresslevel=9) as zf:
        for k, v in arrays.items():
            with zf.open(k + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(v), allow_pickle=False)


def main():
    only = set(sys.argv[1:])
    for name, kw in GOLDEN_SCENARIOS:
        if only and name not in only:
            continue
        cfg, init, tape = make_scenario(**kw)
        rec = run_reference(cfg, init, tape)
        out = {"cfg_json": np.array(cfg_to_json(cfg)), "scenario_json": np.array(json.dumps(kw))}
        for k, v in init.items():
            out["init_" + k] = np.asarray(v)
        for k, v in tape.items():
            out["tape_" + k] = np.asarray(v)
        out.update(rec)
        path = os.path.join(HERE, name + ".npz")
        save_npz(path, out)
        print("%-18s T=%3d hits=%4d anthill_food=%6.1f explored=%6d  %7.1f KB" % (
            name, tape["rot"].shape[0], int(rec["wall_hits"]), float(rec["final_anthill_food"]),
            int(rec["final_explored"].sum()), os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()


# ---------------------------------------------------------------------------------------------------------
# Generator fixtures: the reference's EnvironmentGenerator.generate (environment_generator.py:52-106) with its
# own CirclesGenerator (map_generators.py:28-46) for walls and food, for a few seeds / sizes.
GEN_CASES = [
    ("gen_200_s1000", dict(w=200, h=200, n_ants=50, n_rocks=0, walls=(10, 5, 15), food=(20, 5, 10), seed=1000)),
    ("gen_200_s1001", dict(w=200, h=200, n_ants=50, n_rocks=0, walls=(10, 5, 15), food=(20, 5, 10), seed=1001)),
    ("gen_96x64_s7", dict(w=96, h=64, n_ants=33, n_rocks=0, walls=(6, 3, 9), food=(8, 3, 6), seed=7)),
    ("gen_rocks_s5", dict(w=128, h=128, n_ants=40, n_rocks=5, walls=(8, 5, 12), food=(10, 4, 8), seed=5)),
]


def make_generator_fixtures():
    ref = ref_harness.load_reference()
    for name, c in GEN_CASES:
        ref.gen.n_rocks = c["n_rocks"]     # works around the bare name at environment_generator.py:83-84 (Q17)
        reward = ref.rewards.All_Rewards(1, 2, 10, 1, 3)
        api = ref.api.RLApi(reward, 1, 1, 40 / 180 * np.pi, 0.05, 0.5)
        g = ref.gen.EnvironmentGenerator(c["w"], c["h"], c["n_ants"], 2, c["n_rocks"],
                                         ref.maps.CirclesGenerator(*c["food"]), ref.maps.CirclesGenerator(*c["walls"]),
                                         100, seed=c["seed"])
        env = g.generate(api)
        objs = {"pheros": []}
        for o in env.objects:
            n = type(o).__name__
            if n == "Anthill": objs["anthill"] = o
            elif n == "Walls": objs["walls"] = o
            elif n == "Food": objs["food"] = o
            elif n == "CircleObstacles": objs["rocks"] = o
            elif n == "Ants": objs["ants"] = o
            elif n == "Pheromone": objs["pheros"].append(o)
        st = ref_harness.export_state(env, api, objs)
        out = {"case_json": np.array(json.dumps(c)),
               "channels": np.array([type(o).__name__ for o in api.perceived_objects])}
        for k, v in st.items():
            out["state_" + k] = np.asarray(v)
        out["mask"] = api.perception_mask.astype(np.uint8)
        out["fwd_delta"] = np.float64(api.perception_fwd_delta)
        out["radius"] = np.int64(api.perception_radius)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        print("%-18s walls=%5d food=%5d  %6.1f KB" % (name, int(st["walls"].sum()), int(st["food"].sum()),
                                                      os.path.getsize(path) / 1024))


def make_mainloop_fixture():
    """main.py's loop on the reference's own generator with the reference's own (untaped) global-RNG collision
    noise: generate(seed=1000) -> agent.initialize (activate_all_pheromones(10)) -> np.random.seed(777) ->
    observation -> 80 x [step(random actions); env.update()]."""
    ref = ref_harness.load_reference()
    ref_harness.set_diffuse(ref, 0, 0.001)
    ref.gen.n_rocks = 0
    reward = ref.rewards.All_Rewards(1, 2, 10, 1, 3)
    api = ref.api.RLApi(reward, 1, 1, 40 / 180 * np.pi, 0.05, 0.5)
    g = ref.gen.EnvironmentGenerator(200, 200, 50, 2, 0, ref.maps.CirclesGenerator(20, 5, 10),
                                     ref.maps.CirclesGenerator(10, 5, 15), 80, seed=1000)
    env = g.generate(api)
    api.ants.activate_all_pheromones(np.ones((50, 2)) * 10)         # collect_agent.py:100-102
    np.random.seed(777)
    act = np.random.RandomState(4242)
    ref.walls_proxy.noise_row = None
    out = {"obs": [], "agent_state": [], "reward": [], "done": [], "xyt": [], "holding": [], "anthill_food": []}
    obs0, as0, st0 = api.observation()
    anthill = [o for o in env.objects if type(o).__name__ == "Anthill"][0]
    for t in range(80):
        rot = act.randint(0, 3, 50) - 1
        ph = act.randint(0, 3, 50)
        obs, ast, rew, done = api.step(rot, ph)
        ref.walls_proxy.noise_row = None
        env.update()
        out["obs"].append(obs.astype(np.float32)); out["agent_state"].append(ast); out["reward"].append(np.array(rew, dtype=float))
        out["done"].append(done); out["xyt"].append(api.ants.ants.copy()); out["holding"].append(api.ants.holding.copy())
        out["anthill_food"].append(float(anthill.food))
    path = os.path.join(HERE, "mainloop_s1000.npz")
    np.savez_compressed(path, obs0=obs0.astype(np.float32), agent_state0=as0, state0=st0,
                        final_phero=np.stack([o.phero for o in env.objects if type(o).__name__ == "Pheromone"]),
                        final_food=[o for o in env.objects if type(o).__name__ == "Food"][0].qte,
                        final_explored=reward.explored_map.astype(np.uint8), next_global_draw=np.random.random(),
                        **{k: np.array(v) for k, v in out.items()})
    print("mainloop_s1000 %.1f KB, delivered food %.0f" % (os.path.getsize(path) / 1024, out["anthill_food"][-1]))


if __name__ == "__main__" and (not sys.argv[1:] or "gen" in sys.argv[1:]):
    make_generator_fixtures()
if __name__ == "__main__" and (not sys.argv[1:] or "mainloop" in sys.argv[1:]):
    make_mainloop_fixture()


# ---------------------------------------------------------------------------------------------------------
# Snapshot fixture: the file main.py:136-147 writes for the viewer -- pickle.dump of the list of
# env.save_state() copies (environment.py:36-40), one per step -- from the unmodified reference with rocks.
ARL_CASE = dict(w=48, h=40, n_ants=12, n_rocks=2, walls=(4, 3, 6), food=(6, 3, 5), seed=7, steps=10,
                np_seed=99, action_seed=5)


def make_episode_arl_fixture():
    import pickle
    c = ARL_CASE
    ref = ref_harness.load_reference()
    ref_harness.set_diffuse(ref, 0, 0.001)
    ref.gen.n_rocks = c["n_rocks"]                                   # Q17 workaround, as above
    reward = ref.rewards.All_Rewards(1, 2, 10, 1, 3)
    api = ref.api.RLApi(reward, 1, 1, 40 / 180 * np.pi, 0.05, 0.5)
    g = ref.gen.EnvironmentGenerator(c["w"], c["h"], c["n_ants"], 2, c["n_rocks"],
                                     ref.maps.CirclesGenerator(*c["food"]), ref.maps.CirclesGenerator(*c["walls"]),
                                     c["steps"], seed=c["seed"])
    env = g.generate(api)
    api.ants.activate_all_pheromones(np.ones((c["n_ants"], 2)) * 10)
    np.random.seed(c["np_seed"])
    act = np.random.RandomState(c["action_seed"])
    ref.walls_proxy.noise_row = None
    api.observation()
    states = []
    for t in range(c["steps"]):
        rot = act.randint(0, 3, c["n_ants"]) - 1
        ph = act.randint(0, 3, c["n_ants"])
        api.step(rot, ph)
        ref.walls_proxy.noise_row = None
        env.update()
        states.append(env.save_state())                              # main.py:136-137
    path = os.path.join(HERE, "episode_s7.arl")
    with open(path, "wb") as f:
        pickle.dump(states, f)                                       # main.py:139-147 (first episode: [] + states)
    with open(os.path.join(HERE, "episode_s7.json"), "w") as f:
        json.dump(c, f)
    print("episode_s7.arl %.1f KB, %d states" % (os.path.getsize(path) / 1024, len(states)))


if __name__ == "__main__" and (not sys.argv[1:] or "arl" in sys.argv[1:]):
    make_episode_arl_fixture()


# ---------------------------------------------------------------------------------------------------------
# Long-horizon fixture (BASELINE.json configs[0]: the default 200x200 map with 50 ants driven by random actions for
# 1000 steps): per-step summaries instead of full observations keep it small.
LONG_KW = dict(seed=1001, w=200, h=200, n_ants=50, steps=1000, n_walls=10, n_food=20, wall_r=(5, 15), food_r=(5, 10))
LONG_SNAP_EVERY = 250


def long_summary(obs, agent_state, reward, st, cfg):
    """One row of per-step summary; shared by the recorder and by tests/test_oracle_golden.py."""
    cells = st["x"].astype(np.int64) * cfg["h"] + st["y"].astype(np.int64)
    weights = np.arange(1, cells.size + 1, dtype=np.int64)
    return np.array([st["x"].sum(), st["y"].sum(), st["theta"].sum(), np.asarray(reward, dtype=float).sum(),
                     st["holding"].sum(), float(st["anthill_food"]), float(np.asarray(st["explored"]).sum()),
                     st["phero"][0].sum(), st["phero"][1].sum(), st["food"].sum(), np.asarray(obs, dtype=float).sum(),
                     np.asarray(agent_state, dtype=float).sum(), float((cells * weights).sum()),
                     float(np.asarray(st["mandibles"]).astype(np.int64).sum()),
                     float(np.asarray(st["reward_state"]).astype(np.int64).sum())])


def make_long_fixture():
    cfg, init, tape = make_scenario(**LONG_KW)
    ref = ref_harness.load_reference()
    ref_harness.set_diffuse(ref, cfg["diffuse_factor"], cfg["evap_factor"])
    env, api, objs = ref_harness.build_env(ref, cfg, init)
    objs["ants"].activate_all_pheromones(np.asarray(init["activation"], dtype=float))
    api.observation()
    T = tape["rot"].shape[0]
    rows, snaps = [], {}
    for t in range(T):
        obs, agent_state, reward, done = api.step(tape["rot"][t].astype(np.int64), tape["ph"][t].astype(np.int64))
        ref_harness.run_update(ref, env, tape["noise"][t])
        st = ref_harness.export_state(env, api, objs)
        rows.append(long_summary(obs, agent_state, reward, st, cfg))
        if (t + 1) % LONG_SNAP_EVERY == 0:
            snaps["snap%d" % (t + 1)] = np.stack([st["x"], st["y"], st["theta"], st["holding"],
                                                   st["mandibles"].astype(float), st["reward_state"].astype(float)])
    final = ref_harness.export_state(env, api, objs)
    out = {"cfg_json": np.array(cfg_to_json(cfg)), "scenario_json": np.array(json.dumps(LONG_KW)),
           "t_summary": np.array(rows), "done_last": np.bool_(done), "wall_hits": np.int64(ref.walls_proxy.hits)}
    ref.walls_proxy.hits = 0
    out.update(snaps)
    for k in ("x", "y", "theta", "holding", "mandibles", "reward_state", "phero", "food", "explored", "anthill_food",
              "rewards", "rw_prev_dist", "rw_holding_prev", "timestep"):
        out["final_" + k] = np.asarray(final[k])
    path = os.path.join(HERE, "long_200_s1001.npz")
    np.savez_compressed(path, **out)
    print("long_200_s1001 T=%d hits=%d anthill_food=%.0f explored=%d  %.1f KB" % (
        T, int(out["wall_hits"]), float(final["anthill_food"]), int(final["explored"].sum()), os.path.getsize(path) / 1024))


if __name__ == "__main__" and (not sys.argv[1:] or "long" in sys.argv[1:]):
    make_long_fixture()
