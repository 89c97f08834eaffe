#!/usr/bin/env python
"""Cost of starting new episodes on a used handle, at the cfg4 shard (512 envs of 1024^2) and at cfg3 (4096 envs of
256^2), the benchmark's CirclesGenerator maps:

* today's reset: bench.generate_states_parallel (a fork pool over generate_state), stack_states, and the complete-state
  import a used handle needs (walls, food, zero pheromone planes, zero explored, the ants), to a device synchronise;
* the device reset: the host draws (generate_episode, one process and a fork pool), ants_generate_env_maps (disc upload,
  k_reset_maps, bookkeeping) and the per-ant import, and BatchedEnvironmentGenerator.reset end to end.  k_reset_maps is
  timed by CUDA events (the `reset` kernel family, warmed up, median over --launches calls); its bytes written over
  that time are set against the 6546 GB/s copy peak of SURVEY.md section 6.

Both resets are made from the same seeds and their states compared (two envs, every key).  Prints one JSON line per
workload; the GPU name and power limit are read in the same run.

With --walls perlin the workload's walls are the reference's default PerlinGenerator() (main.py:75) instead, and the
script reports reset(perlin="host") end to end (host noise over every cell, complete import), the host draws
(generate_episode(perlin=True)), the generate_env_maps call, the Perlin kernel's CUDA-event median next to the Circles
kernel's median on the same window in the same run (the yardstick of the Perlin kernel), the memset yardstick, the
per-ant import, reset(perlin="device") end to end, and a two-env comparison of the two paths.

    python scripts/reset_bench.py [--workloads cfg4 cfg3] [--launches 25] [--walls {circles,perlin}]
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402

import bench         # noqa: E402

COPY_PEAK_GBS = 6546.0          # SURVEY.md section 6: device-to-device copy peak measured on the B200


def _draw_chunk(args):
    wl, first, n = args
    from antsrl_b200.generator import generate_episode
    g = bench.make_generator(wl, 1000)
    return [generate_episode(g.w, g.h, g.n_ants, g.n_pheromones, g.n_rocks, g.food_generator, g.walls_generator,
                             seed=g.seed_base + first + e) for e in range(n)]


def draws_parallel(wl, n_envs):
    nproc = max(1, min(os.cpu_count() or 1, 32, n_envs))
    per = (n_envs + nproc - 1) // nproc
    jobs = [(wl, s, min(per, n_envs - s)) for s in range(0, n_envs, per)]
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        parts = pool.map(_draw_chunk, jobs)
    return [e for p in parts for e in p]


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as ex:   # (the numbers are still printed; the card's settings are then unknown)
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % ex
    return info


def wall(fn):
    t = time.perf_counter()
    r = fn()
    return time.perf_counter() - t, r


def run(name, launches):
    import torch
    from antsrl_b200 import BatchedAnts
    from antsrl_b200.generator import generate_episode, stack_states
    wl = bench.WORKLOADS[name]
    E, N, W, H, P = wl["envs_per_gpu"], wl["n_ants"], wl["w"], wl["h"], wl["n_phero"]
    gen = bench.make_generator(wl, 1000)
    b = BatchedAnts(gen.cfg, E, evap_mode="lazy", record="compact8")
    res = {"workload": name, "envs": E, "map": [W, H], "ants_per_env": N, "record": "compact8"}

    # ---- the device reset, piece by piece
    g = gen
    res["draws_one_process_s"], eps = wall(lambda: [generate_episode(g.w, g.h, N, P, g.n_rocks, g.food_generator,
                                                                     g.walls_generator, seed=g.seed_base + e)
                                                    for e in range(E)])
    res["draws_fork_pool_s"], eps_p = wall(lambda: draws_parallel(wl, E))
    assert all(np.array_equal(a["wall_discs"], c["wall_discs"]) for a, c in zip(eps, eps_p))
    hill = np.stack([e["anthill_xyr"] for e in eps])
    wd, fd = np.stack([e["wall_discs"] for e in eps]), np.stack([e["food_discs"] for e in eps])
    for _ in range(3):                                         # warm-up
        b.generate_env_maps(hill, wd, fd)
    b.set_profiling(True)
    call_s, kern_ms = [], []
    for _ in range(launches):
        b.reset_kernel_ms()
        dt, _ = wall(lambda: b.generate_env_maps(hill, wd, fd))
        call_s.append(dt)
        ms, n = b.kernel_ms()["reset"]
        assert n == 1
        kern_ms.append(ms)
    b.set_profiling(False)
    res["generate_env_maps_call_s_median"] = statistics.median(call_s)
    res["kernel_ms_median"] = statistics.median(kern_ms)
    res["kernel_ms_min_max"] = [min(kern_ms), max(kern_ms)]
    res["kernel_launches_timed"] = launches
    rec_bytes = 8
    wp, hp = -(-W // 16) * 16, -(-H // 16) * 16
    written = E * wp * hp * rec_bytes
    res["kernel_bytes_written"] = written
    res["kernel_GBps"] = written / (res["kernel_ms_median"] / 1e3) / 1e9
    res["kernel_share_of_copy_peak"] = res["kernel_GBps"] / COPY_PEAK_GBS
    # a write-only yardstick of the same size in the same run: cudaMemsetAsync (torch zero_) by CUDA events
    buf = torch.empty(written, dtype=torch.uint8, device="cuda")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms_set = []
    for k in range(13):
        ev[0].record()
        buf.zero_()
        ev[1].record()
        torch.cuda.synchronize()
        if k >= 3:
            ms_set.append(ev[0].elapsed_time(ev[1]))
    del buf
    res["memset_same_bytes_ms_median"] = statistics.median(ms_set)
    res["memset_GBps"] = written / (res["memset_same_bytes_ms_median"] / 1e3) / 1e9
    res["kernel_share_of_memset"] = res["kernel_GBps"] / res["memset_GBps"]
    ants = {k: np.stack([e[k] for e in eps]) for k in ("x", "y", "theta", "seed", "rw_prev_dist")}
    if g.n_rocks:
        ants.update({k: np.stack([e[k] for e in eps]) for k in ("rock_centers", "rock_radii", "rock_weights")})
    ants.update(prev_x=ants["x"], prev_y=ants["y"], prev_theta=ants["theta"], holding=np.zeros((E, N)),
                rewards=np.zeros((E, N)), rw_holding_prev=np.zeros((E, N)), mandibles=np.zeros((E, N), np.uint8),
                reward_state=np.zeros((E, N), np.uint8), anthill_food=np.zeros(E),
                activation=np.full((E, N, P), 10.0), timestep=1, rw_alias=True, act_bool=False)
    t_ant = []
    for _ in range(5):
        dt, _ = wall(lambda: b.import_state(ants))
        t_ant.append(dt)
    res["per_ant_import_s_median"] = statistics.median(t_ant)
    res["device_reset_total_fork_pool_s"] = (res["draws_fork_pool_s"] + res["generate_env_maps_call_s_median"]
                                             + res["per_ant_import_s_median"])
    t_reset = []
    for _ in range(3):
        dt, _ = wall(lambda: (gen.reset(b, gen.seed_base), b.synchronize()))
        t_reset.append(dt)
    res["reset_call_one_process_s_median"] = statistics.median(t_reset)
    dev_state = b.export_state(envs=(0, 2))

    # ---- today's reset: host planes for every env, complete-state import
    dt_gen, states = wall(lambda: bench.generate_states_parallel(wl, 1000, 0, E))
    dt_stack, st = wall(lambda: stack_states(states, "all"))
    del states
    st.update(phero=np.zeros((E, P, W, H)), explored=np.zeros((E, W, H), np.uint8),
              holding=np.zeros((E, N)), rewards=np.zeros((E, N)), rw_holding_prev=np.zeros((E, N)),
              mandibles=np.zeros((E, N), np.uint8), reward_state=np.zeros((E, N), np.uint8), anthill_food=np.zeros(E),
              activation=np.full((E, N, P), 10.0), act_bool=False)
    host_bytes = sum(v.nbytes for v in st.values() if isinstance(v, np.ndarray))
    dt_imp, _ = wall(lambda: (b.import_state(st), b.synchronize()))
    del st
    res["today_generate_states_parallel_s"] = dt_gen
    res["today_stack_states_s"] = dt_stack
    res["today_import_s"] = dt_imp
    res["today_import_bytes"] = host_bytes
    res["today_total_s"] = dt_gen + dt_stack + dt_imp
    host_state = b.export_state(envs=(0, 2))
    same = all(np.array_equal(v, host_state[k]) if isinstance(v, np.ndarray) else v == host_state[k]
               for k, v in dev_state.items())
    res["device_reset_equals_host_reset"] = bool(same)
    res["speedup_total_fork_pool"] = res["today_total_s"] / res["device_reset_total_fork_pool_s"]
    res["speedup_reset_call"] = res["today_total_s"] / res["reset_call_one_process_s_median"]
    res["speedup_vs_import_only"] = dt_imp / (res["generate_env_maps_call_s_median"] + res["per_ant_import_s_median"])
    b.close()
    torch.cuda.synchronize()
    return res


def _kernel_median(b, launches, hill, walls, food):
    """generate_env_maps on the whole batch: the call's wall time and the `reset` family's CUDA-event time, medians over
    `launches` calls after 3 warm-up calls."""
    for _ in range(3):
        b.generate_env_maps(hill, walls, food)
    b.set_profiling(True)
    call_s, kern_ms = [], []
    for _ in range(launches):
        b.reset_kernel_ms()
        dt, _ = wall(lambda: b.generate_env_maps(hill, walls, food))
        call_s.append(dt)
        ms, n = b.kernel_ms()["reset"]
        assert n == 1
        kern_ms.append(ms)
    b.set_profiling(False)
    return statistics.median(call_s), statistics.median(kern_ms), [min(kern_ms), max(kern_ms)]


def run_perlin(name, launches):
    import torch
    from antsrl_b200 import BatchedAnts
    from antsrl_b200.generator import PerlinGenerator, generate_episode
    wl = bench.WORKLOADS[name]
    E, N, W, H, P = wl["envs_per_gpu"], wl["n_ants"], wl["w"], wl["h"], wl["n_phero"]
    circles = bench.make_generator(wl, 1000)
    gen = bench.make_generator(wl, 1000)
    gen.walls_generator = PerlinGenerator()
    b = BatchedAnts(gen.cfg, E, evap_mode="lazy", record="compact8")
    res = {"workload": name, "walls": "PerlinGenerator()", "envs": E, "map": [W, H], "ants_per_env": N,
           "record": "compact8"}
    g = gen
    res["draws_one_process_s"], eps = wall(lambda: [generate_episode(g.w, g.h, N, P, g.n_rocks, g.food_generator,
                                                                     g.walls_generator, seed=g.seed_base + e,
                                                                     perlin=True) for e in range(E)])
    hill = np.stack([e["anthill_xyr"] for e in eps])
    layer, fd = g.walls_generator.layer(np.stack([e["wall_perlin"] for e in eps])), np.stack([e["food_discs"] for e in eps])
    res["generate_env_maps_call_s_median"], res["perlin_kernel_ms_median"], res["perlin_kernel_ms_min_max"] = \
        _kernel_median(b, launches, hill, layer, fd)
    c_eps = [generate_episode(W, H, N, P, circles.n_rocks, circles.food_generator, circles.walls_generator,
                              seed=circles.seed_base + e) for e in range(E)]
    _, res["circles_kernel_ms_median"], res["circles_kernel_ms_min_max"] = _kernel_median(
        b, launches, np.stack([e["anthill_xyr"] for e in c_eps]), np.stack([e["wall_discs"] for e in c_eps]),
        np.stack([e["food_discs"] for e in c_eps]))
    res["kernel_launches_timed"] = launches
    res["perlin_over_circles_kernel"] = res["perlin_kernel_ms_median"] / res["circles_kernel_ms_median"]
    res["perlin_kernel_within_2x_of_circles"] = bool(res["perlin_over_circles_kernel"] <= 2.0)
    written = E * (-(-W // 16) * 16) * (-(-H // 16) * 16) * 8
    res["kernel_bytes_written"] = written
    buf = torch.empty(written, dtype=torch.uint8, device="cuda")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms_set = []
    for k in range(13):
        ev[0].record()
        buf.zero_()
        ev[1].record()
        torch.cuda.synchronize()
        if k >= 3:
            ms_set.append(ev[0].elapsed_time(ev[1]))
    del buf
    res["memset_same_bytes_ms_median"] = statistics.median(ms_set)
    ants = {k: np.stack([e[k] for e in eps]) for k in ("x", "y", "theta", "seed", "rw_prev_dist")}
    if g.n_rocks:
        ants.update({k: np.stack([e[k] for e in eps]) for k in ("rock_centers", "rock_radii", "rock_weights")})
    ants.update(prev_x=ants["x"], prev_y=ants["y"], prev_theta=ants["theta"], holding=np.zeros((E, N)),
                rewards=np.zeros((E, N)), rw_holding_prev=np.zeros((E, N)), mandibles=np.zeros((E, N), np.uint8),
                reward_state=np.zeros((E, N), np.uint8), anthill_food=np.zeros(E),
                activation=np.full((E, N, P), 10.0), timestep=1, rw_alias=True, act_bool=False)
    t_ant = []
    for _ in range(5):
        dt, _ = wall(lambda: b.import_state(ants))
        t_ant.append(dt)
    res["per_ant_import_s_median"] = statistics.median(t_ant)
    t_reset = []
    for _ in range(3):
        dt, path = wall(lambda: (gen.reset(b, gen.seed_base, perlin="device"), b.synchronize())[0])
        assert path == "device"
        t_reset.append(dt)
    res["device_reset_one_process_s_median"] = statistics.median(t_reset)
    dev_state = b.export_state(envs=(0, 2))
    dt_host, path = wall(lambda: (gen.reset(b, gen.seed_base), b.synchronize())[0])
    assert path == "host"
    res["host_reset_one_process_s"] = dt_host
    host_state = b.export_state(envs=(0, 2))
    res["device_reset_equals_host_reset"] = bool(all(
        np.array_equal(v, host_state[k]) if isinstance(v, np.ndarray) else v == host_state[k]
        for k, v in dev_state.items()))
    res["speedup_reset_call"] = dt_host / res["device_reset_one_process_s_median"]
    b.close()
    torch.cuda.synchronize()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["cfg4", "cfg3"], choices=sorted(bench.WORKLOADS))
    ap.add_argument("--launches", type=int, default=25, help="timed k_reset_maps launches (median)")
    ap.add_argument("--walls", choices=["circles", "perlin"], default="circles",
                    help="the workload's CirclesGenerator walls, or the reference's default PerlinGenerator()")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("reset_bench.py measures on a CUDA device; there is none")
    info = gpu_info()
    for name in a.workloads:
        r = (run if a.walls == "circles" else run_perlin)(name, max(a.launches, 20))
        r.update(info)
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
