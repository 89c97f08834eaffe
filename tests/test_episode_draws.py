"""The random draws of a new episode without its planes (antsrl_b200.generator.generate_episode, the input of
ants_generate_env_maps): pinned to the reference's recordings (tests/golden/gen_*.npz) through a host stamp of the
discs, consuming the global RNGs exactly like generate_state, and the choice between the device and the host path of
BatchedEnvironmentGenerator.reset."""
import glob
import json
import os
import random

import numpy as np
import pytest

from golden_io import GOLDEN_DIR
from antsrl_b200.generator import (BatchedEnvironmentGenerator, CirclesGenerator, PerlinGenerator, disc_area,
                                   disc_inside, generate_episode, generate_state)

CASES = sorted(glob.glob(os.path.join(GOLDEN_DIR, "gen_*.npz")))


def _stamp(w, h, ep, food_gen, walls_gen):
    """What ants_generate_env_maps writes, on the host: walls = union of the wall discs outside the anthill disc, food =
    1 on the union of the food discs outside the walls."""
    walls = walls_gen.stamp(w, h, ep["wall_discs"])
    walls[disc_area(w, h, *ep["anthill_xyr"].tolist())] = False
    food = food_gen.stamp(w, h, ep["food_discs"]).astype(float) * (1 - walls)
    return walls.astype(np.uint8), food


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_episode_draws_match_reference(path):
    z = np.load(path)
    c = json.loads(str(z["case_json"]))
    fg, wg = CirclesGenerator(*c["food"]), CirclesGenerator(*c["walls"])
    ep = generate_episode(c["w"], c["h"], c["n_ants"], 2, c["n_rocks"], fg, wg, seed=c["seed"])
    assert ep is not None
    assert ep["wall_discs"].dtype == np.int32 and ep["wall_discs"].shape == (c["walls"][0], 3)
    assert ep["food_discs"].shape == (c["food"][0], 3)
    walls, food = _stamp(c["w"], c["h"], ep, fg, wg)
    assert np.array_equal(walls, z["state_walls"])
    assert np.array_equal(food, z["state_food"])
    for k in ("anthill_xyr", "x", "y", "theta", "seed"):
        assert np.array_equal(ep[k], z["state_" + k]), k
    if c["n_rocks"]:
        for k in ("rock_centers", "rock_radii", "rock_weights"):
            assert np.array_equal(ep[k], z["state_" + k]), k
    assert len(CASES) >= 4


@pytest.mark.parametrize("n_rocks", [0, 5])
def test_episode_draws_leave_the_rngs_where_generate_state_does(n_rocks):
    args = (200, 160, 40, 2, n_rocks, CirclesGenerator(20, 5, 10), CirclesGenerator(10, 5, 15))
    st = generate_state(*args, seed=77)
    after_state = (random.random(), np.random.random())
    ep = generate_episode(*args, seed=77)
    after_episode = (random.random(), np.random.random())
    assert after_state == after_episode
    from antsrl_b200.generator import stack_states
    assert np.array_equal(ep["rw_prev_dist"], stack_states([st])["rw_prev_dist"][0])


def test_draw_discs_is_generate():
    g = CirclesGenerator(30, 5, 15)
    random.seed(3)
    discs = g.draw_discs(128, 96)
    nxt = random.random()
    random.seed(3)
    m = g.generate(128, 96)
    assert random.random() == nxt
    assert np.array_equal(m, g.stamp(128, 96, discs))
    assert disc_inside(discs, 128, 96)
    assert not disc_inside(np.array([[3, 50, 4]]), 128, 96)
    assert not disc_inside(np.array([[60, 92, 4]]), 128, 96)
    assert not disc_inside(np.array([[60, 50, -1]]), 128, 96)


class _FakeBatch:
    """Records what reset hands to the binding (no device needed)."""

    def __init__(self, E, env_id_base=0):
        self.E, self.env_id_base = E, env_id_base
        self.calls = []

    def generate_env_maps(self, anthill_xyr, wall_discs, food_discs, envs=None):
        self.calls.append(("maps", envs, anthill_xyr, wall_discs, food_discs))

    def import_state(self, state, envs=None):
        self.calls.append(("import", envs, state))


class _DuckCircles:
    """A user generator with CirclesGenerator's behaviour but not its type: it draws from the global RNG itself."""

    def __init__(self, *a):
        self.g = CirclesGenerator(*a)

    def generate(self, w, h):
        return self.g.generate(w, h)


def test_reset_of_a_map_smaller_than_a_disc_is_the_host_path():
    """A disc wider than the map has no disc form; the reference's own stamp fails on such a map (an index past the
    edge), and so does reset, before anything reaches the handle."""
    food, walls = CirclesGenerator(6, 5, 10), CirclesGenerator(4, 14, 15)
    gen = BatchedEnvironmentGenerator(24, 24, 8, 2, 0, food, walls, max_steps=10)
    random.seed(1)
    assert not disc_inside(walls.draw_discs(24, 24), 24, 24)
    b = _FakeBatch(2)
    with pytest.raises(IndexError):
        generate_state(24, 24, 8, 2, 0, food, walls, seed=7)
    with pytest.raises(IndexError):
        gen.reset(b, 7)
    assert b.calls == []


@pytest.mark.parametrize("case", ["perlin", "duck"])
def test_reset_takes_the_host_path(case):
    w = h = 64
    food, walls = CirclesGenerator(6, 5, 10), CirclesGenerator(4, 5, 15)
    if case == "perlin":
        walls = PerlinGenerator(scale=22.0, density=0.1)
    else:
        food = _DuckCircles(6, 5, 10)
    gen = BatchedEnvironmentGenerator(w, h, 8, 2, 0, food, walls, max_steps=10)
    b = _FakeBatch(4, env_id_base=8)
    assert gen.reset(b, 500, envs=(1, 2)) == "host"
    assert [c[0] for c in b.calls] == ["import"]
    _, envs, st = b.calls[0]
    assert envs == (1, 2)
    ref = [generate_state(w, h, 8, 2, 0, food, walls, seed=500 + 8 + 1 + e) for e in range(2)]
    for k in ("walls", "food", "anthill_xyr", "x", "y", "theta", "seed"):
        assert np.array_equal(st[k], np.stack([r[k] for r in ref])), k
    assert not st["phero"].any() and not st["explored"].any()
    assert "timestep" not in st and "act_bool" not in st      # a window keeps the batch's scalars


def test_reset_takes_the_device_path():
    food, walls = CirclesGenerator(6, 5, 10), CirclesGenerator(4, 5, 15)
    gen = BatchedEnvironmentGenerator(96, 80, 8, 2, 3, food, walls, max_steps=10)
    b = _FakeBatch(3, env_id_base=4)
    assert gen.reset(b, 100) == "device"
    assert [c[0] for c in b.calls] == ["maps", "import"]
    _, envs, hill, wd, fd = b.calls[0]
    assert envs == (0, 3) and hill.shape == (3, 3) and wd.shape == (3, 4, 3) and fd.shape == (3, 6, 3)
    st = b.calls[1][2]
    assert "walls" not in st and "food" not in st and "phero" not in st
    ref = [generate_state(96, 80, 8, 2, 3, food, walls, seed=100 + 4 + e) for e in range(3)]
    for k in ("x", "y", "theta", "seed", "rock_centers", "rock_radii", "rock_weights"):
        assert np.array_equal(st[k], np.stack([r[k] for r in ref])), k
    assert np.array_equal(hill, np.stack([r["anthill_xyr"] for r in ref]))
    assert st["timestep"] == 1 and st["rw_alias"] is True and st["act_bool"] is False
    assert np.all(st["activation"] == 10.0)
