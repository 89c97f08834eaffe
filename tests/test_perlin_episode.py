"""The draws of Perlin map layers (PerlinGenerator.draw_offsets, generate_episode(..., perlin=True)) and the device path
of BatchedEnvironmentGenerator.reset(..., perlin="device"), without a device: the offsets are exactly generate's RNG
calls, a host stamp of the draws rebuilds generate_state's planes, and reset hands the right layers to the binding."""
import ctypes
import random

import numpy as np
import pytest

from antsrl_b200.generator import (BatchedEnvironmentGenerator, CirclesGenerator, PerlinGenerator, disc_area,
                                   generate_episode, generate_state)
from antsrl_b200.perlin import PerlinLayer
from test_episode_draws import _DuckCircles, _FakeBatch

PARAMS = [dict(), dict(scale=0.7, density=0.0, octaves=1), dict(scale=33.0, density=-0.1, octaves=5, persistence=0.6,
                                                                    lacunarity=2.3), dict(scale=-13.0, density=0.2)]


@pytest.mark.parametrize("kw", PARAMS, ids=["default", "one-octave", "five-octaves", "negative-scale"])
def test_draw_offsets_is_generate(kw):
    g = PerlinGenerator(**kw)
    random.seed(11)
    offs = g.draw_offsets()
    nxt = random.random()
    random.seed(11)
    m = g.generate(90, 70)
    assert random.random() == nxt
    assert offs.dtype == np.int32 and offs.shape == (2,)
    assert np.array_equal(m, g.stamp(90, 70, offs))
    lay = g.layer([offs, offs])
    assert isinstance(lay, PerlinLayer) and lay.offsets.shape == (2, 2) and lay.offsets.dtype == np.int32
    assert (lay.scale, lay.density, lay.octaves) == (g.scale, g.density, g.octaves)


def _stamp(w, h, ep, food_gen, walls_gen):
    """What ants_generate_env_maps_ex writes, on the host: the walls layer outside the anthill disc, food = 1 where the
    food layer is set and the cell is not a wall."""
    def layer(name, g):
        return g.stamp(w, h, ep[name + "_perlin"]) if name + "_perlin" in ep else g.stamp(w, h, ep[name + "_discs"])
    walls = layer("wall", walls_gen)
    walls[disc_area(w, h, *ep["anthill_xyr"].tolist())] = False
    food = layer("food", food_gen).astype(float) * (1 - walls)
    return walls.astype(np.uint8), food


MIXES = {"perlin-walls": (CirclesGenerator(20, 5, 10), PerlinGenerator()),
         "perlin-food": (PerlinGenerator(scale=15.0, density=0.1), CirclesGenerator(10, 5, 15)),
         "both-perlin": (PerlinGenerator(scale=9.0, density=0.2, octaves=3), PerlinGenerator(density=-0.05))}


@pytest.mark.parametrize("n_rocks", [0, 5])
@pytest.mark.parametrize("mix", sorted(MIXES))
def test_episode_with_perlin_layers_is_generate_state(mix, n_rocks):
    food, walls = MIXES[mix]
    args = (200, 160, 40, 2, n_rocks, food, walls)
    st = generate_state(*args, seed=77)
    after_state = (random.random(), np.random.random())
    ep = generate_episode(*args, seed=77, perlin=True)
    after_episode = (random.random(), np.random.random())
    assert after_state == after_episode
    assert ("wall_perlin" in ep) == (type(walls) is PerlinGenerator)
    assert ("food_perlin" in ep) == (type(food) is PerlinGenerator)
    for name in ("wall", "food"):
        if name + "_perlin" in ep:
            assert ep[name + "_perlin"].dtype == np.int32 and ep[name + "_perlin"].shape == (2,)
            assert name + "_discs" not in ep
    w, f = _stamp(200, 160, ep, food, walls)
    assert np.array_equal(w, st["walls"]) and np.array_equal(f, st["food"])
    assert st["walls"].any() and st["food"].any()
    keys = ("anthill_xyr", "x", "y", "theta", "seed") + (("rock_centers", "rock_radii", "rock_weights") if n_rocks else ())
    for k in keys:
        assert np.array_equal(ep[k], st[k]), k


def test_episode_without_perlin_option_keeps_the_host_form():
    food, walls = CirclesGenerator(6, 5, 10), PerlinGenerator()
    random.seed(5)
    before = random.getstate()
    assert generate_episode(64, 64, 8, 2, 0, food, walls, seed=None) is None
    assert random.getstate() == before                    # nothing drawn
    assert generate_episode(64, 64, 8, 2, 0, _DuckCircles(6, 5, 10), walls, seed=3, perlin=True) is None


@pytest.mark.parametrize("envs", [None, (1, 2)])
def test_reset_with_perlin_on_the_device(envs):
    w, h = 96, 80
    food, walls = CirclesGenerator(6, 5, 10), PerlinGenerator(scale=22.0, density=0.1)
    gen = BatchedEnvironmentGenerator(w, h, 8, 2, 3, food, walls, max_steps=10)
    b = _FakeBatch(4, env_id_base=8)
    assert gen.reset(b, 100, envs=envs, perlin="device") == "device"
    assert [c[0] for c in b.calls] == ["maps", "import"]
    env0, n = (0, 4) if envs is None else envs
    _, got_envs, hill, wl, fd = b.calls[0]
    assert got_envs == (env0, n)
    assert isinstance(wl, PerlinLayer) and wl.offsets.shape == (n, 2) and fd.shape == (n, 6, 3)
    assert (wl.scale, wl.density, wl.octaves, wl.persistence, wl.lacunarity) == (22.0, 0.1, 2, 0.5, 2.0)
    seeds = [100 + 8 + env0 + e for e in range(n)]
    ref = [generate_state(w, h, 8, 2, 3, food, walls, seed=s) for s in seeds]
    eps = [generate_episode(w, h, 8, 2, 3, food, walls, seed=s, perlin=True) for s in seeds]
    assert np.array_equal(wl.offsets, np.stack([ep["wall_perlin"] for ep in eps]))
    assert np.array_equal(fd, np.stack([ep["food_discs"] for ep in eps]))
    assert np.array_equal(hill, np.stack([r["anthill_xyr"] for r in ref]))
    for e, ep in enumerate(eps):                              # the layers stamp generate_state's planes
        wp, fp = _stamp(w, h, ep, food, walls)
        assert np.array_equal(wp, ref[e]["walls"]) and np.array_equal(fp, ref[e]["food"])
    st = b.calls[1][2]
    assert "walls" not in st and "food" not in st and "phero" not in st
    for k in ("x", "y", "theta", "seed", "rock_centers", "rock_radii", "rock_weights"):
        assert np.array_equal(st[k], np.stack([r[k] for r in ref])), k
    assert ("timestep" in st) == (envs is None)


def test_reset_with_perlin_food_and_walls_on_the_device():
    food, walls = PerlinGenerator(scale=9.0, density=0.2, octaves=3), PerlinGenerator()
    gen = BatchedEnvironmentGenerator(64, 64, 8, 2, 0, food, walls, max_steps=10)
    b = _FakeBatch(2)
    assert gen.reset(b, 7, perlin="device") == "device"
    _, _, _, wl, fl = b.calls[0]
    assert isinstance(wl, PerlinLayer) and isinstance(fl, PerlinLayer)
    assert fl.octaves == 3 and wl.octaves == 2


def test_duck_typed_layer_takes_the_host_path_with_perlin_on_the_device():
    food, walls = _DuckCircles(6, 5, 10), PerlinGenerator(density=0.1)
    gen = BatchedEnvironmentGenerator(64, 64, 8, 2, 0, food, walls, max_steps=10)
    b = _FakeBatch(2)
    assert gen.reset(b, 500, perlin="device") == "host"
    assert [c[0] for c in b.calls] == ["import"]
    with pytest.raises(ValueError):
        gen.reset(b, 500, perlin="gpu")


def test_perlin_layer_struct_size():
    from antsrl_b200 import _cabi
    # AntsPerlinLayer: pointer, 2 doubles, 2 int32, 2 doubles (by hand from include/antsrl_b200.h)
    assert ctypes.sizeof(_cabi.AntsPerlinLayer) == 8 + 2 * 8 + 2 * 4 + 2 * 8
    assert _cabi.AntsPerlinLayer.octaves.offset == 24 and _cabi.AntsPerlinLayer.persistence.offset == 32
