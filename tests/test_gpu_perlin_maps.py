"""Perlin map layers on the device (ants_generate_env_maps_ex, ants_perlin_noise): the noise field equals perlin.py bit
for bit, and a reset with perlin="device" leaves a handle exactly where the host path (generate_state through
perlin.py, then a complete import) leaves it, before and after running the episode."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_episode_reset import ARMS, RUN, SHAPES, _assert_same_state, _gen, _iterate, _used_handle

pytestmark = pytest.mark.gpu

FIELD_CASES = {   # name: (w, h, offsets, scale, octaves, persistence, lacunarity)
    "1024-default": (1024, 1024, [(123, -456), (-9876, 5), (0, 0)], 22.0, 2, 0.5, 2.0),
    "200-extreme-offsets": (200, 200, [(-10000, 10000), (10000, -10000), (-10000, -10000)], 22.0, 2, 0.5, 2.0),
    "333x97-5-octaves": (333, 97, [(5, 7), (-300, 4000)], 22.0, 5, 0.6, 2.3),
    "256-scale-0.7-one-octave": (256, 256, [(10, -10), (-7777, 31)], 0.7, 1, 0.5, 2.0),
    "300x500-scale-300": (300, 500, [(1, 2), (9000, -9000)], 300.0, 3, 0.35, 1.7),
    "scale-minus-13": (128, 96, [(50, -50), (-1234, 4321)], -13.0, 2, 0.5, 2.0),
    "12-octaves-repeat-2^21": (96, 64, [(9999, -9999), (-3, 17)], 22.0, 12, 0.5, 2.0),
    "7-octaves-lacunarity-3": (100, 90, [(3, 4), (-5000, 2500)], 3.3, 7, 0.9, 3.0),
}


@pytest.mark.parametrize("case", sorted(FIELD_CASES))
def test_device_field_equals_perlin_py(case):
    from antsrl_b200.perlin import perlin_noise_device, perlin_noise_generator
    w, h, offs, scale, octaves, pers, lac = FIELD_CASES[case]
    got = perlin_noise_device(w, h, np.array(offs), scale=scale, octaves=octaves, persistence=pers,
                              lacunarity=lac).cpu().numpy()
    assert got.shape == (len(offs), w, h) and got.dtype == np.float32
    for k, (ox, oy) in enumerate(offs):
        ref = perlin_noise_generator(w, h, ox, oy, scale=scale, octaves=octaves, persistence=pers,
                                     lacunarity=lac).astype(np.float32)
        a, b = ref + np.float32(0), got[k] + np.float32(0)        # zero signs normalised
        bad = np.flatnonzero(a.view(np.int32) != b.view(np.int32))
        assert bad.size == 0, "%s, offsets %r: %d cells differ, first %r: %r != %r" % (
            case, (ox, oy), bad.size, np.unravel_index(bad[0], a.shape), b.flat[bad[0]], a.flat[bad[0]])
        assert np.ptp(ref) > 0.1


def _perlin_gen(w, h, n_ants, n_rocks=0, walls=None, food=None, **cfg_kw):
    """The generator of test_gpu_episode_reset with PerlinGenerator() walls (or `walls`) and, given, `food`."""
    from antsrl_b200.generator import PerlinGenerator
    gen = _gen(w, h, n_ants, n_rocks, walls=PerlinGenerator() if walls is None else walls, **cfg_kw)
    if food is not None:
        gen.food_generator = food
    return gen


def _main_py_gen():
    """main.py:74-75: 200 x 200, 50 ants, CirclesGenerator(20, 5, 10) food and the default PerlinGenerator walls."""
    from antsrl_b200.generator import BatchedEnvironmentGenerator, CirclesGenerator, PerlinGenerator
    return BatchedEnvironmentGenerator(200, 200, 50, 2, 0, CirclesGenerator(20, 5, 10), PerlinGenerator(),
                                       max_steps=2000, seed_base=1000)


def _density_on_a_noise_value():
    """Walls whose density is a noise value of env 0's map: the strict > decides the cells that hold it."""
    from antsrl_b200.generator import PerlinGenerator, generate_episode
    from antsrl_b200.perlin import perlin_noise_generator
    gen = _perlin_gen(200, 200, 50)
    ep = generate_episode(200, 200, 50, 2, 0, gen.food_generator, PerlinGenerator(), seed=gen.seed_base, perlin=True)
    field = perlin_noise_generator(200, 200, *ep["wall_perlin"].tolist())
    v = np.sort(field.ravel())[field.size // 2]
    assert np.count_nonzero(field == v) >= 1
    gen.walls_generator = PerlinGenerator(density=float(v))
    return gen


def _perlin_arm(name):
    from antsrl_b200.generator import CirclesGenerator, PerlinGenerator
    if name == "main.py":
        return _main_py_gen()
    if name == "perlin-food":
        return _perlin_gen(200, 200, 50, walls=CirclesGenerator(15, 5, 15), food=PerlinGenerator(scale=15.0, density=0.1))
    if name == "both-perlin":
        return _perlin_gen(200, 200, 50, food=PerlinGenerator(scale=9.0, density=0.2, octaves=3),
                           walls=PerlinGenerator(density=-0.05))
    if name == "density-on-a-value":
        return _density_on_a_noise_value()
    raise KeyError(name)


CASES = [(a, "200x50") for a in ARMS] + [(a, "256x256") for a in ("compact8-lazy", "f64-lazy", "f64-diffuse")] \
        + [("compact8-lazy", "1024x1024")] \
        + [(a, "special") for a in ("main.py", "perlin-food", "both-perlin", "density-on-a-value")]


@pytest.mark.parametrize("arm,shape", CASES, ids=["%s-%s" % c for c in CASES])
def test_perlin_reset_of_a_used_handle_equals_a_new_handle(arm, shape):
    import torch
    if shape == "special":
        gen, (gkw, kw), E = _perlin_arm(arm), ARMS["compact8-lazy"], 6
        n_ants = gen.n_ants
    else:
        gkw, kw = ARMS[arm]
        w, h, n_ants, n_rocks, E = SHAPES[shape]
        if arm.endswith("1100"):
            n_ants = 1100
        gen = _perlin_gen(w, h, n_ants, n_rocks, **gkw)
    b = _used_handle(gen, E, kw)
    assert gen.reset(b, gen.seed_base, perlin="device") == "device"
    a = gen.generate(E, **kw)                           # the host path through perlin.py
    st = a.export_state(keys=("walls", "food"))
    assert st["walls"].any() and st["food"].any()
    _assert_same_state(a, b, "after the reset")
    _iterate(b, RUN, 77, ref=a)
    _assert_same_state(a, b, "after %d iterations" % RUN)
    b2 = _used_handle(gen, E, kw)
    gen.reset(b2, gen.seed_base, perlin="device")
    a2 = gen.generate(E, **kw)
    g = torch.Generator(device="cuda").manual_seed(5)
    rot = torch.randint(-1, 2, (RUN, E, n_ants), dtype=torch.int8, device="cuda", generator=g)
    ph = torch.randint(0, 3, (RUN, E, n_ants), dtype=torch.int8, device="cuda", generator=g)
    ra, rb = a2.rollout(rot, ph), b2.rollout(rot, ph)
    for x, y in zip(ra, rb):
        assert torch.equal(x, y)
    _assert_same_state(a2, b2, "after a rollout of %d steps" % RUN)
    for x in (a, b, a2, b2):
        x.close()


@pytest.mark.parametrize("record", ["compact8", "f64"])
def test_perlin_window_reset_equals_the_host_path(record):
    gen = _perlin_gen(120, 104, 40, 3)
    kw = dict(evap_mode="lazy", record=record)
    dev, host = gen.generate(4, **kw), gen.generate(4, **kw)
    _iterate(dev, 9, 11, ref=host)
    assert gen.reset(dev, 4242, envs=(1, 2), perlin="device") == "device"
    assert gen.reset(host, 4242, envs=(1, 2)) == "host"
    _assert_same_state(host, dev, "after the window reset")
    for t in range(15):
        _iterate(dev, 1, 300 + t, ref=host)
        _assert_same_state(host, dev, "after update %d" % (10 + t))
    dev.close()
    host.close()


def test_fresh_handle_with_perlin_reset_equals_generate():
    from antsrl_b200 import BatchedAnts
    gen = _main_py_gen()
    kw = dict(evap_mode="lazy", record="compact8")
    b = BatchedAnts(gen.cfg, 5, **kw)
    assert gen.reset(b, gen.seed_base, perlin="device") == "device"
    a = gen.generate(5, **kw)
    _assert_same_state(a, b, "after the reset")
    _iterate(b, 20, 3, ref=a)
    _assert_same_state(a, b, "after 20 iterations")
    a.close()
    b.close()


def test_sharded_perlin_resets_equal_one_handle():
    from antsrl_b200 import BatchedAnts
    E = 6
    gen = _perlin_gen(128, 128, 64, 4)
    kw = dict(evap_mode="lazy", record="compact8", rng_seed=3)
    whole = BatchedAnts(gen.cfg, E, **kw)
    shards = [BatchedAnts(gen.cfg, E // 2, env_id_base=s * E // 2, **kw) for s in range(2)]
    for x in [whole] + shards:
        assert gen.reset(x, 600, perlin="device") == "device"
    for t in range(12):
        ow = whole.step(*whole.sample_actions(40 + t))
        for s, x in enumerate(shards):
            o = x.step(*x.sample_actions(40 + t))
            sl = slice(s * E // 2, (s + 1) * E // 2)
            assert all(np.array_equal(o[k].cpu().numpy(), ow[k][sl].cpu().numpy()) for k in range(3)), t
        for x in [whole] + shards:
            x.update(None)
    sw = whole.export_state()
    parts = [x.export_state() for x in shards]
    for k, v in sw.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, np.concatenate([p[k] for p in parts])), k
    for x in [whole] + shards:
        x.close()


def _discs():
    hill = np.ascontiguousarray([[30, 30, 4], [20, 40, 3]], dtype=np.int32)
    wd = np.ascontiguousarray([[[10, 10, 5], [40, 45, 8]], [[50, 50, 6], [20, 12, 7]]], dtype=np.int32)
    fd = np.ascontiguousarray([[[40, 12, 5]], [[12, 40, 5]]], dtype=np.int32)
    return hill, wd, fd


def test_ex_with_two_disc_layers_equals_generate_env_maps():
    gen = _gen(64, 64, 16)
    kw = dict(evap_mode="lazy", record="compact8")
    a, b = gen.generate(2, **kw), gen.generate(2, **kw)
    _iterate(a, 5, 1, ref=b)
    hill, wd, fd = _discs()
    i32 = C.POINTER(C.c_int32)
    assert a.lib.ants_generate_env_maps(a._h, 0, 2, hill.ctypes.data_as(i32), 2, wd.ctypes.data_as(i32), 1,
                                        fd.ctypes.data_as(i32)) == 0
    assert b.lib.ants_generate_env_maps_ex(b._h, 0, 2, hill.ctypes.data_as(i32), 2, wd.ctypes.data_as(i32), None, 1,
                                           fd.ctypes.data_as(i32), None) == 0
    _assert_same_state(a, b, "after the two calls")
    assert a.export_state(keys=("walls",))["walls"].any()
    _iterate(a, 10, 2, ref=b)
    a.close()
    b.close()


def test_bad_perlin_arguments_are_rejected_and_leave_the_handle():
    from antsrl_b200 import AntsError
    from antsrl_b200.perlin import PerlinLayer, perlin_layer_struct, perlin_noise_device
    gen = _gen(64, 64, 16)
    b = gen.generate(2, evap_mode="lazy", record="compact8")
    _iterate(b, 5, 1)
    before = b.export_state()
    hill, wd, fd = _discs()
    i32 = C.POINTER(C.c_int32)
    good = PerlinLayer(np.array([[3, 4], [-5, 6]]), 22.0, 0.05, 2, 0.5, 2.0)

    def call(wl=None, n_w=0, fl=None, n_f=1, null_offsets=False, env0=0, n=2):
        keep = []
        ptrs = []
        for lay in (wl, fl):
            if lay is None:
                ptrs.append(None)
                continue
            s, offs = perlin_layer_struct(lay)
            keep.append(offs)
            if null_offsets:
                s.offsets = None
            ptrs.append(C.pointer(s))
        return b.lib.ants_generate_env_maps_ex(b._h, env0, n, hill.ctypes.data_as(i32), n_w, wd.ctypes.data_as(i32),
                                               ptrs[0], n_f, fd.ctypes.data_as(i32), ptrs[1])
    bad = {
        "window past the batch": dict(wl=good, env0=1),
        "empty window": dict(wl=good, n=0),
        "octaves 0": dict(wl=good._replace(octaves=0)),
        "octaves 33": dict(wl=good._replace(octaves=33)),
        "scale 0": dict(wl=good._replace(scale=0.0)),
        "scale inf": dict(wl=good._replace(scale=float("inf"))),
        "scale nan": dict(wl=good._replace(scale=float("nan"))),
        "persistence nan": dict(wl=good._replace(persistence=float("nan"))),
        "persistence beyond float": dict(wl=good._replace(persistence=1e300)),
        "lacunarity inf": dict(wl=good._replace(lacunarity=float("inf"))),
        "wall layer with discs and Perlin": dict(wl=good, n_w=2),
        "food layer with discs and Perlin": dict(fl=good, n_w=2, n_f=1),
        "NULL offsets": dict(wl=good, null_offsets=True),
        "period 0 (lacunarity 0)": dict(wl=good._replace(lacunarity=0.0)),
        "period past 2^31": dict(wl=good._replace(lacunarity=3e6)),
        "coordinate past 2^31": dict(wl=good._replace(offsets=np.array([[10000, 0], [0, 0]]), scale=1.0,
                                                      lacunarity=2e6)),
        "coordinate past 2^31, one octave": dict(wl=good._replace(scale=1e-8, octaves=1)),
    }
    for what, kw in bad.items():
        assert call(**kw) == -1, what               # ANTS_E_ARG
    fd_out = np.ascontiguousarray([[[40, 12, 5]], [[12, 62, 5]]], dtype=np.int32)
    s, offs = perlin_layer_struct(good)
    assert b.lib.ants_generate_env_maps_ex(b._h, 0, 2, hill.ctypes.data_as(i32), 0, wd.ctypes.data_as(i32),
                                           C.pointer(s), 1, fd_out.ctypes.data_as(i32), None) == -1
    after = b.export_state()
    for k, v in before.items():
        assert (np.array_equal(v, after[k]) if isinstance(v, np.ndarray) else v == after[k]), k
    assert call(wl=good) == 0
    assert call(wl=good, fl=good._replace(density=0.2), n_f=0) == 0
    for kw in (dict(octaves=0), dict(scale=0.0), dict(lacunarity=float("nan"))):
        args = dict(scale=22.0, octaves=2, persistence=0.5, lacunarity=2.0)
        args.update(kw)
        with pytest.raises(AntsError):
            perlin_noise_device(32, 32, np.array([[1, 2]]), **args)
    b.close()
