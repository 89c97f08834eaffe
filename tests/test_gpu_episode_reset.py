"""New episodes on an existing handle: BatchedEnvironmentGenerator.reset writes the maps on the device
(ants_generate_env_maps) from the generator's draws.  A reset of a used handle must leave it exactly where a new
handle built by `generate()` from the same seeds starts, and both must then run the same episode bit for bit."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DIRTY = 40        # iterations that leave pheromone, explored, held food, moved rocks and the anthill store behind
RUN = 150         # iterations after the reset (past the 7-bit generation fold of the compact records at ~124)


def _gen(w, h, n_ants, n_rocks=0, seed_base=1000, walls=None, **cfg_kw):
    from antsrl_b200.generator import BatchedEnvironmentGenerator, CirclesGenerator
    n_w, n_f = max(4, w * h // 2600), max(6, w * h // 3300)     # cfg4: 400 / 320 discs on 1024 x 1024
    return BatchedEnvironmentGenerator(w, h, n_ants, 2, n_rocks, CirclesGenerator(n_f, 5, 10),
                                       walls if walls is not None else CirclesGenerator(n_w, 5, 15),
                                       max_steps=2000, seed_base=seed_base, **cfg_kw)


def _iterate(b, n, seed, ref=None):
    """n x [step(device-drawn random actions); update(Philox)]; with `ref`, the same on it and every output equal."""
    import torch
    for t in range(n):
        rot, ph = b.sample_actions(seed + t)
        o = b.step(rot, ph)
        if ref is not None:
            r = ref.step(rot, ph)
            for k, name in enumerate(("obs", "agent_state", "reward")):
                assert torch.equal(o[k], r[k]), "%s differs at iteration %d" % (name, t)
            assert o[3] == r[3]
            ref.update(None)
        b.update(None)


def _assert_same_state(a, b, what, phero_rtol=0.0):
    sa, sb = a.export_state(), b.export_state()
    for k in sa:
        if k == "phero" and phero_rtol:
            np.testing.assert_allclose(sb[k], sa[k], rtol=phero_rtol, atol=0, err_msg="%s: phero" % what)
        elif isinstance(sa[k], np.ndarray):
            assert sa[k].dtype == sb[k].dtype and np.array_equal(sa[k], sb[k]), "%s: %s differs" % (what, k)
        else:
            assert sa[k] == sb[k], "%s: %s %r != %r" % (what, k, sa[k], sb[k])


def _used_handle(gen, E, kw):
    """A handle of the same configuration with another episode run on it for DIRTY iterations."""
    b = _with_seed(gen, gen.seed_base + 7919).generate(E, **kw)
    _iterate(b, DIRTY, 555)
    st = b.export_state(keys=("phero", "explored", "holding", "anthill_food", "rock_centers"))
    assert st["phero"].any() and st["explored"].any()
    return b


ARMS = {   # name: (generator kwargs, generate() kwargs)
    "compact8-lazy": ({}, dict(evap_mode="lazy", record="compact8")),
    "compact-lazy": ({}, dict(evap_mode="lazy", record="compact")),
    "f64-lazy": ({}, dict(evap_mode="lazy", record="f64")),
    "f64-tiles": ({}, dict(evap_mode="tiles", record="f64")),
    "f64-dense": ({}, dict(evap_mode="dense", record="f64")),
    "f64-diffuse": (dict(diffuse_factor=0.02, evap_factor=0.01), dict(evap_mode="dense", record="f64")),
    "compact8-lazy-1100": ({}, dict(evap_mode="lazy", record="compact8")),
}
SHAPES = {"200x50": (200, 200, 50, 0, 8), "256x256": (256, 256, 256, 0, 4), "1024x1024": (1024, 1024, 1024, 64, 2)}
CASES = [(a, "200x50") for a in ARMS] + [(a, "256x256") for a in ("compact8-lazy", "f64-lazy", "f64-dense", "f64-diffuse")] \
        + [("compact8-lazy", "1024x1024")]


@pytest.mark.parametrize("arm,shape", CASES, ids=["%s-%s" % c for c in CASES])
def test_reset_of_a_used_handle_equals_a_new_handle(arm, shape):
    import torch
    gkw, kw = ARMS[arm]
    w, h, n_ants, n_rocks, E = SHAPES[shape]
    if arm.endswith("1100"):
        n_ants = 1100                    # flat kernels on a lazy field: the owner plane
    gen = _gen(w, h, n_ants, n_rocks, **gkw)
    b = _used_handle(gen, E, kw)
    assert gen.reset(b, gen.seed_base) == "device"
    a = gen.generate(E, **kw)
    _assert_same_state(a, b, "after the reset")
    _iterate(b, RUN, 77, ref=a)
    _assert_same_state(a, b, "after %d iterations" % RUN)
    # the same episode again through ants_rollout (device tapes, Philox noise)
    b2 = _used_handle(gen, E, kw)
    gen.reset(b2, gen.seed_base)
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
def test_window_reset_equals_the_host_import(record, monkeypatch):
    """envs [1, 3) of 4 get a new episode at iteration 9, once written on the device and once imported as complete
    host states (the path tests/test_gpu_parity.py checks against the oracle); the other envs run on untouched, and
    both handles agree after every step and update."""
    import antsrl_b200.generator as G
    gen = _gen(120, 104, 40, 3)
    kw = dict(evap_mode="lazy", record=record)
    dev, host = gen.generate(4, **kw), gen.generate(4, **kw)
    _iterate(dev, 9, 11, ref=host)
    assert gen.reset(dev, 4242, envs=(1, 2)) == "device"
    with monkeypatch.context() as m:
        m.setattr(G, "generate_episode", lambda *a, **k: None)
        assert gen.reset(host, 4242, envs=(1, 2)) == "host"
    _assert_same_state(host, dev, "after the window reset")
    st = dev.export_state(keys=("timestep", "anthill_xyr"))
    assert st["timestep"] == 10
    for t in range(15):
        _iterate(dev, 1, 300 + t, ref=host)
        _assert_same_state(host, dev, "after update %d" % (10 + t))
    dev.close()
    host.close()


@pytest.mark.parametrize("record,lead", [("compact8", 254 - 4), ("f64", 4094 - 4)])
def test_reset_next_to_the_lazy_fold(record, lead):
    """A handle reset a few updates before k_lazy_fold re-bases its plain pheromone values (every 254 / 4094 updates):
    the fold runs on the reset handle and not on the new one.  Outputs and state agree bit for bit except the pheromone
    values, which the fold rounds once more (8-byte records keep a plain value as f32: 6e-8 relative; f64: 1e-13)."""
    import torch
    gen = _gen(96, 80, 48, 2)
    kw = dict(evap_mode="lazy", record=record)
    b = gen.generate(2, **kw)
    b.rollout(None, None, n_steps=lead)
    gen.reset(b, 31)
    a = _with_seed(gen, 31).generate(2, **kw)
    _assert_same_state(a, b, "after the reset")
    b.reset_kernel_ms()
    a.reset_kernel_ms()
    tol = 1e-6 if record == "compact8" else 1e-12
    for t in range(20):
        rot, ph = a.sample_actions(900 + t)
        oa, ob = a.step(rot, ph), b.step(rot, ph)
        assert torch.equal(oa[1], ob[1]) and torch.equal(oa[2], ob[2]), "iteration %d" % t
        torch.testing.assert_close(ob[0], oa[0], rtol=tol, atol=1e-7)
        a.update(None)
        b.update(None)
    assert b.kernel_ms()["evaporate"][1] == 1 and a.kernel_ms()["evaporate"][1] == 0     # the fold fell in the window
    _assert_same_state(a, b, "after the fold", phero_rtol=tol)
    a.close()
    b.close()


def _with_seed(gen, seed_base):
    from antsrl_b200.generator import BatchedEnvironmentGenerator
    g = BatchedEnvironmentGenerator.__new__(BatchedEnvironmentGenerator)
    g.__dict__.update(gen.__dict__)
    g.seed_base = seed_base
    return g


def test_sharded_resets_equal_one_handle():
    from antsrl_b200 import BatchedAnts
    E = 6
    gen = _gen(128, 128, 64, 4)
    kw = dict(evap_mode="lazy", record="compact8", rng_seed=3)
    whole = BatchedAnts(gen.cfg, E, **kw)
    shards = [BatchedAnts(gen.cfg, E // 2, env_id_base=s * E // 2, **kw) for s in range(2)]
    for x in [whole] + shards:
        assert gen.reset(x, 600) == "device"
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


def test_host_path_with_perlin_walls_equals_a_new_handle():
    from antsrl_b200.generator import PerlinGenerator
    gen = _gen(96, 96, 40, 2, walls=PerlinGenerator(scale=22.0, density=0.1))
    kw = dict(evap_mode="lazy", record="compact8")
    b = _used_handle(gen, 3, kw)
    assert gen.reset(b, gen.seed_base) == "host"
    a = gen.generate(3, **kw)
    _assert_same_state(a, b, "after the reset")
    _iterate(b, 30, 8, ref=a)
    _assert_same_state(a, b, "after 30 iterations")
    a.close()
    b.close()


def test_bad_arguments_are_rejected_and_leave_the_handle():
    gen = _gen(64, 64, 16)
    b = gen.generate(2, evap_mode="lazy", record="compact8")
    _iterate(b, 5, 1)
    before = b.export_state()
    i32 = C.POINTER(C.c_int32)

    def call(env0, n, hill, wd, fd, n_w=None, n_f=None):
        hill, wd, fd = (np.ascontiguousarray(x, dtype=np.int32) for x in (hill, wd, fd))
        return b.lib.ants_generate_env_maps(b._h, env0, n, hill.ctypes.data_as(i32),
                                            wd.shape[1] if n_w is None else n_w, wd.ctypes.data_as(i32),
                                            fd.shape[1] if n_f is None else n_f, fd.ctypes.data_as(i32))
    hill = np.array([[30, 30, 4], [20, 40, 3]])
    wd = np.array([[[10, 10, 5]], [[50, 50, 6]]])
    fd = np.array([[[40, 12, 5]], [[12, 40, 5]]])
    bad = {
        "window before the batch": (-1, 2, hill, wd, fd),
        "window past the batch": (1, 2, hill, wd, fd),
        "empty window": (0, 0, hill, wd, fd),
        "negative anthill radius": (0, 2, [[30, 30, -1], [20, 40, 3]], wd, fd),
        "negative wall radius": (0, 2, hill, [[[10, 10, -2]], [[50, 50, 6]]], fd),
        "wall disc past the left edge": (0, 2, hill, [[[3, 10, 5]], [[50, 50, 6]]], fd),
        "food disc past the far edge": (0, 2, hill, wd, [[[40, 12, 5]], [[12, 59, 5]]]),
        "negative wall count": (0, 2, hill, wd, fd, -1, None),
        "negative food count": (0, 2, hill, wd, fd, None, -3),
    }
    for what, args in bad.items():
        assert call(*args) == -1, what          # ANTS_E_ARG
    after = b.export_state()
    for k, v in before.items():
        assert (np.array_equal(v, after[k]) if isinstance(v, np.ndarray) else v == after[k]), k
    assert call(0, 2, hill, wd, fd) == 0
    b.close()
