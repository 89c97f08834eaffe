#!/usr/bin/env python
"""main.py's loop with everything resident in HBM (SURVEY.md section 8-f rows 2 and 3).

observation -> epsilon-greedy action (a torch MLP with the collect agents' two heads, agents/collect_agent.py:
20-58, random-initialised here; the exploration branch drawn by ants_sample_actions) -> step -> replay-memory ingest
-> update, for E environments at once.  Observations, actions, rewards and the replay memory never cross PCIe; the
only host traffic per step is kernel launches.  PyTorch is plumbing (the MLP and the ring-buffer copies).

    python examples/on_device_loop.py [--envs 512] [--steps 50] [--workload cfg4] [--episodes K] [--walls perlin]

With --episodes K > 1 an episode lasts --steps steps, and when `done` arrives every env starts a new one
(main.py:66-79) through BatchedEnvironmentGenerator.reset, which writes the new maps on the device; the share of the
wall time spent in those resets is printed.  With --walls perlin the walls are main.py's default PerlinGenerator()
(main.py:75) instead of the workload's discs; its maps are written on the device too (reset(..., perlin="device")).
"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch         # noqa: E402

import bench         # noqa: E402
from antsrl_b200 import BatchedAnts                      # noqa: E402
from antsrl_b200.generator import PerlinGenerator, stack_states   # noqa: E402
from antsrl_b200.replay import DeviceReplayMemory        # noqa: E402
from antsrl_b200.device_loop import DeviceActionSelector  # noqa: E402


class TwoHeadPolicy(torch.nn.Module):                    # the shape of CollectModel (collect_agent.py:20-58)
    def __init__(self, obs_dim, agent_dim, rotations=3, pheromones=3, hidden=64):
        super().__init__()
        self.l1 = torch.nn.Linear(obs_dim + agent_dim, hidden)
        self.l2 = torch.nn.Linear(hidden, hidden)
        self.rot = torch.nn.Linear(hidden, rotations)
        self.ph = torch.nn.Linear(hidden, pheromones)

    def forward(self, obs, agent_state):
        x = torch.cat((obs.flatten(1), agent_state), dim=1)
        x = torch.relu(self.l2(torch.relu(self.l1(x))))
        return self.rot(x), self.ph(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg4", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--epsilon", type=float, default=0.3)
    ap.add_argument("--replay", type=int, default=1 << 20)
    ap.add_argument("--episodes", type=int, default=1, help="episodes of --steps steps each (1: one episode, no reset)")
    ap.add_argument("--walls", choices=["circles", "perlin"], default="circles",
                    help="the workload's CirclesGenerator walls, or main.py's default PerlinGenerator()")
    a = ap.parse_args()
    wl = bench.WORKLOADS[a.workload]
    E, N = a.envs, wl["n_ants"]
    gen = bench.make_generator(wl, a.steps + 10 if a.episodes <= 1 else a.steps)
    perlin = "device" if a.walls == "perlin" else "host"
    env = BatchedAnts(gen.cfg, E, evap_mode="lazy", record="compact8")
    if a.walls == "perlin":
        gen.walls_generator = PerlinGenerator()                                  # main.py:75
        gen.reset(env, gen.seed_base, perlin=perlin)                             # = gen.generate(E), maps on the device
    else:
        states = bench.generate_states_parallel(wl, a.steps + 10, 0, E)
        env.import_state(stack_states(states, "all"))
        env.activate_all_pheromones(np.ones((E, N, wl["n_phero"])) * 10.0)      # agent.initialize
    C = len(gen.cfg["channels"])
    policy = TwoHeadPolicy(49 * C, 2).cuda().half()
    mem = DeviceReplayMemory(a.replay, (7, 7, C), (2,), 2)
    selector = DeviceActionSelector(env, a.epsilon, seed=1234)
    obs, ast, _, _ = env.observe()                                               # main.py:88
    obs, ast = obs.clone(), ast.clone()
    total_reward = torch.zeros((), dtype=torch.float64, device="cuda")
    warm = 5                                                                     # cuBLAS / allocator warm-up, untimed
    n_iter = a.steps + warm if a.episodes <= 1 else a.steps * a.episodes
    reset_s, episode = 0.0, 0
    for t in range(n_iter):
        if t == warm:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            total_reward.zero_()
        with torch.no_grad():                                                    # collect_agent.py:161-177
            q_rot, q_ph = policy(obs.reshape(E * N, -1).half(), ast.reshape(E * N, 2).half())
            rot, ph, _ = selector.select(q_rot, q_ph)                            # argmax, or explore, per environment
        new_obs, new_ast, rew, done = env.step(rot, ph)                          # main.py:98
        mem.extend(obs, ast, (rot, ph), rew, new_obs, new_ast, done)             # main.py:102
        env.update(None)                                                         # main.py:131
        total_reward += rew.sum()
        obs, ast = new_obs.clone(), new_ast.clone()
        if done and a.episodes > 1 and episode + 1 < a.episodes:                # main.py:66-79: a new environment
            episode += 1
            r0 = time.perf_counter()
            gen.reset(env, gen.seed_base + episode * E, perlin=perlin)           # (reset synchronises the stream)
            obs, ast, _, _ = env.observe()
            obs, ast = obs.clone(), ast.clone()
            torch.cuda.synchronize()
            reset_s += time.perf_counter() - r0
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    n_steps = n_iter - warm
    print("on-device loop: %d envs x %d ants x %d steps in %.3f s = %.3e ant-steps/s (policy forward + replay ingest "
          "included), mean reward/ant-step %.4f, replay fill %d" %
          (E, N, n_steps, dt, E * N * n_steps / dt, float(total_reward) / (E * N * n_steps), len(mem)))
    if a.episodes > 1:
        print("%d episodes: %d resets took %.3f s, %.1f %% of the wall time" % (episode + 1, episode, reset_s, 100.0 * reset_s / dt))
    env.close()


if __name__ == "__main__":
    main()
