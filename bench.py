#!/usr/bin/env python
"""bench.py -- ant-steps/s of the AntsRL environment step loop on B200 (contract in the task brief).

One "step" = one pass of the hot path over the whole batch: RLApi.step(actions_t) followed by Environment.update()
(obs, agent_state and reward materialised in HBM every step), on synthetic maps from the drop-in generator
(env e <- seed 1000 + e, actions i.i.d. uniform rot in {-1,0,1}, ph in {0,1,2} from RandomState(12345), in-kernel
Philox collision noise).  value = envs x ants x steps / time, whole job over all ranks (weak scaling: the per-GPU
shard is fixed; N = 8 of the default workload is BASELINE.json configs[3]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg4|cfg3|cfg2] [--envs E] [--evap lazy|tiles|dense]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...      # the UNMODIFIED reference (oracle/_ref) on the host cores

--dump-outputs DIR writes the outputs of the last timed step (obs, agent_state, reward) as DIR/<name>.npy; the inputs
are seeded, so two builds run with the same arguments can be compared output for output.

The timed region is ONE C call (ants_rollout over a device-resident action tape): per step one launch of the perception
kernel and one of the block-per-environment kernel (update_k ; move of step_{k+1}); no Python between the steps.

Extra JSON keys: roofline (dominant kernel vs measured HBM peak; dram_frac = ncu-measured DRAM bytes of the same launch),
late (the same K steps re-timed around step 900 of the episode, ants dispersed), cpu_baseline (the UNMODIFIED reference,
oracle/_ref, on the host cores; bounded sample), e2e (host buffers through the C ABI, copies inside the timed region),
e2e_packed (the observation left in its packed PCIe form), kernels (per-family ms), clocks.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[3] sharded over 8 GPUs: 512 envs per GPU (SURVEY.md section 8-d, cfg 4)
    "cfg4": dict(w=1024, h=1024, n_ants=1024, n_phero=2, n_rocks=64, walls=(400, 5, 15), food=(320, 5, 10),
                 envs_per_gpu=512, desc="1024x1024 map, 1024 ants/env, 64 rocks, 512 envs per GPU (4096 on 8)"),
    # configs[2]
    "cfg3": dict(w=256, h=256, n_ants=256, n_phero=2, n_rocks=0, walls=(16, 5, 15), food=(26, 5, 10),
                 envs_per_gpu=4096, desc="256x256 map, 256 ants/env, 4096 envs per GPU"),
    # configs[1]
    "cfg2": dict(w=200, h=200, n_ants=50, n_phero=2, n_rocks=0, walls=(10, 5, 15), food=(20, 5, 10),
                 envs_per_gpu=1024, desc="reference default 200x200 map, 50 ants/env, 1024 envs per GPU"),
}


def make_generator(wl, steps):
    from antsrl_b200.generator import BatchedEnvironmentGenerator, CirclesGenerator
    return BatchedEnvironmentGenerator(wl["w"], wl["h"], wl["n_ants"], wl["n_phero"], wl["n_rocks"],
                                       CirclesGenerator(*wl["food"]), CirclesGenerator(*wl["walls"]),
                                       max_steps=steps, seed_base=1000)


def _gen_chunk(args):
    wl, steps, first, n = args
    g = make_generator(wl, steps)
    return g.generate_states(n, first)


def generate_states_parallel(wl, steps, first_env, n_envs):
    nproc = max(1, min(os.cpu_count() or 1, 32, n_envs))
    if nproc == 1 or n_envs < 8:
        return _gen_chunk((wl, steps, first_env, n_envs))
    per = (n_envs + nproc - 1) // nproc
    jobs = [(wl, steps, first_env + s, min(per, n_envs - s)) for s in range(0, n_envs, per)]
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        parts = pool.map(_gen_chunk, jobs)
    return [s for p in parts for s in p]


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML every ~5 ms; nvidia-smi fallback)."""
    SMI_Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flag = lambda name: "Active" if r & getattr(n, name, 0) else "Not Active"
        return [sm, self.max_sm, pw, flag("nvmlClocksThrottleReasonHwSlowdown"),
                flag("nvmlClocksThrottleReasonHwThermalSlowdown"), flag("nvmlClocksThrottleReasonSwThermalSlowdown"),
                flag("nvmlClocksThrottleReasonSwPowerCap")]

    def _run(self):
        while not self._stop.is_set():
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                    self._stop.wait(0.005)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.SMI_Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(str(r[col]).lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(float(r[2]) for r in self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------------------------- CPU baseline
def _reference_available():
    try:
        from oracle import ref_harness
        return ref_harness.reference_available()
    except Exception:
        return False


def _cpu_worker(args):
    """One independent env per process.  kind "reference": the UNMODIFIED reference (oracle/_ref = its modules byte-compiled
    by oracle/build_ref.py, or the checkout) driven through RLApi.step / Environment.update exactly as main.py:88-138
    drives it, its own global-RNG collision noise included.  kind "port": the oracle (numpy restatement)."""
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    wl, env_id, warm, steps, kind = args
    g = make_generator(wl, warm + steps + 1)
    st = g.generate_states(1, env_id)[0]
    N, P = wl["n_ants"], wl["n_phero"]
    rs = np.random.RandomState(12345 + env_id)
    if kind == "reference":
        from oracle import ref_harness
        ref = ref_harness.load_reference()
        ref_harness.set_diffuse(ref, g.cfg["diffuse_factor"], g.cfg["evap_factor"])
        env, api, objs = ref_harness.build_env(ref, g.cfg, st)
        objs["ants"].activate_all_pheromones(np.ones((N, P)) * 10.0)        # agent.initialize, collect_agent.py:100-102
        np.random.seed(777 + env_id)
        api.observation()                                                    # main.py:88
        step = lambda rot, ph, t: (api.step(rot, ph), ref_harness.run_update(ref, env, None))
    else:
        from oracle.antsrl_oracle import OracleEnv, philox_uniform
        env = OracleEnv(g.cfg, st)
        env.activate_all_pheromones(np.ones((N, P)) * 10.0)
        env.observation()
        step = lambda rot, ph, t: (env.step(rot, ph), env.update(philox_uniform(0, env_id, t + 1, N)))
    t0 = None
    for t in range(warm + steps):
        if t == warm:
            t0 = time.perf_counter()
        step(rs.randint(0, 3, N) - 1, rs.randint(0, 3, N), t)
    return time.perf_counter() - t0


def run_cpu_baseline(wl, warm, steps, procs=None):
    procs = procs or (os.cpu_count() or 1)
    kind = "reference" if _reference_available() else "port"
    t_wall = time.perf_counter()
    with mp.get_context("fork").Pool(procs) as pool:
        times = pool.map(_cpu_worker, [(wl, e, warm, steps, kind) for e in range(procs)])
    t_wall = time.perf_counter() - t_wall
    worst = max(times)
    value = procs * wl["n_ants"] * steps / worst
    what = ("the unmodified reference (oracle/_ref: its own RLApi.step + Environment.update, scipy convolve2d, global-RNG "
            "collision noise)" if kind == "reference" else "oracle = numpy port of the reference loop incl. scipy convolve2d")
    return {"value": value, "unit": "ant-steps/s", "cores": procs, "kind": kind,
            "sample": "%d independent envs (one per process, %d processes) x %d timed steps of step()+update() after "
                      "%d warm-up, %dx%d map, %d ants/env, %s" % (procs, procs, steps, warm, wl["w"], wl["h"], wl["n_ants"], what),
            "ms_per_env_step": 1000.0 * float(np.mean(times)) / steps, "wall_s": t_wall}


# ----------------------------------------------------------------------------------------------- roofline
def algorithmic_bytes(fam, wl, E, C, stats):
    """Algorithmic bytes per launch of one kernel family (SURVEY.md section 8-d; stated in DESIGN.md)."""
    N, P, W, H = wl["n_ants"], wl["n_phero"], wl["w"], wl["h"]
    EN = E * N
    if fam == "perceive":       # obs f32 + agent_state + reward out, 49-sample gathers, per-ant state
        per_ant = 49 * C * 4 + 8 + 8 + 49 * (8 * P + 8 + 1 + 1 + 1) + 82
        return EN * per_ant
    if fam == "evaporate":
        if stats.get("evap_mode") == "lazy":
            return 0
        if stats.get("evap_mode") == "tiles":
            return stats["active_tiles"] * 256 * (16 + 1)
        return E * W * H * (16 * P + 1)
    if fam == "move":
        return EN * (48 + 1 + 8 + 2 + 32 + 1 + 8 * P + 2)
    if fam == "collide":
        return EN * (24 + 16 + 1 + 48 + 4 + 2)
    if fam == "deposit":
        return EN * (16 + 4 + 8 * P + 16)
    if fam == "rocks":
        return EN * (16 + 16 + 24) + E * wl["n_rocks"] * 48
    # the block-per-environment kernels do the work of the flat families they replace: the same algorithmic bytes
    if fam == "env_move":
        return algorithmic_bytes("move", wl, E, C, stats)
    if fam == "env_update":
        return sum(algorithmic_bytes(f, wl, E, C, stats) for f in ("collide", "deposit")) + \
            (algorithmic_bytes("rocks", wl, E, C, stats) if wl["n_rocks"] else 0)
    if fam == "env_update_move":
        return algorithmic_bytes("env_update", wl, E, C, stats) + algorithmic_bytes("move", wl, E, C, stats)
    return 0


def ncu_traffic(fam, n_ants):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/latest_traffic.json,
    written by scripts/profile_summary.py: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch).  Used as it
    is when the capture was taken at this batch size, else scaled per ant (and said so)."""
    path = os.path.join(ROOT, "profiles", "latest_traffic.json")
    try:
        d = json.load(open(path))
        if d.get("kernel", "").replace("k_", "") == fam:
            exact = int(d.get("ants", 0)) == int(n_ants)
            return d["dram_bytes_per_ant"] * n_ants, ("ncu capture of this launch size (%s)" % d.get("tag", "") if exact else
                                                      "ncu capture at %d ants, scaled per ant" % int(d.get("ants", 0)))
    except Exception:
        pass
    return None, None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------- --dump-outputs
DUMP_BYTES = 64 * 10 ** 6          # at most this much array data in DIR


def sample_outputs(obs, agent_state, reward):
    """The outputs of one step as a caller of ants_rollout receives them -- obs (E,N,S,S,C) f32, agent_state (E,N,2)
    f32, reward (E,N) f64 -- copied to the host with the env and ant axes flattened (row = env * N + ant).  When all
    ants do not fit in DUMP_BYTES, the rows are a fixed sample: np.sort(RandomState(0).choice(E * N, n, replace=False)),
    the same rows in every array."""
    import torch
    obs, agent_state, reward = (t.reshape(t.shape[0] * t.shape[1], *t.shape[2:]) for t in (obs, agent_state, reward))
    n_all = obs.shape[0]
    per_ant = obs[0].numel() * obs.element_size() + agent_state[0].numel() * agent_state.element_size() + reward.element_size()
    n = min(n_all, (DUMP_BYTES - 3 * 4096) // per_ant)          # 4096: room for each .npy header
    if n < n_all:
        rows = torch.from_numpy(np.sort(np.random.RandomState(0).choice(n_all, n, replace=False))).to(obs.device)
        obs, agent_state, reward = (t.index_select(0, rows) for t in (obs, agent_state, reward))
    return {"obs": obs.cpu().numpy(), "agent_state": agent_state.cpu().numpy(), "reward": reward.cpu().numpy()}


def write_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------- main arms
def make_batch(args, rank=0, device=0):
    """The inputs of one rank, ready for the first step: its envs from the drop-in generator, pheromones activated, the
    first observation taken, and the action tapes (T, E, N) on the device.
    -> (gen, batch, cell record format, rot_tape, ph_tape)."""
    import torch
    from antsrl_b200 import BatchedAnts
    from antsrl_b200.generator import stack_states
    wl = WORKLOADS[args.workload]
    E = args.envs or wl["envs_per_gpu"]
    N = wl["n_ants"]
    K = args.steps
    total_steps = max(args.warmup + 3 * K, args.late_start + K) + 2 * args.e2e_steps + 16
    gen = make_generator(wl, total_steps + 10)
    states = generate_states_parallel(wl, total_steps + 10, rank * E, E)
    record = args.record if args.evap == "lazy" else "f64"
    batch = BatchedAnts(gen.cfg, E, device=device, evap_mode=args.evap, rng_seed=20261018, env_id_base=rank * E,
                        record=record)
    batch.import_state(stack_states(states, gen.cfg["reward_kind"]))
    del states
    batch.activate_all_pheromones(np.ones((E, N, wl["n_phero"])) * 10.0)      # agent.initialize, collect_agent.py:100
    rs = np.random.RandomState(12345 + rank)
    n_tape = max(K, 32)                                                       # the pre-recorded action sequence
    rot_tape = torch.from_numpy((rs.randint(0, 3, size=(n_tape, E, N)) - 1).astype(np.int8)).cuda()
    ph_tape = torch.from_numpy(rs.randint(0, 3, size=(n_tape, E, N)).astype(np.int8)).cuda()
    batch.observe()                                                           # main.py:88
    return gen, batch, record, rot_tape, ph_tape


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep NCCL's version banner off stdout: ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    wl = WORKLOADS[args.workload]
    E = args.envs or wl["envs_per_gpu"]
    N = wl["n_ants"]
    K, W_ = args.steps, args.warmup
    late_start = args.late_start

    t_setup = time.perf_counter()
    gen, batch, record, rot_tape, ph_tape = make_batch(args, rank, local_rank)
    C = len(gen.cfg["channels"])
    n_tape = rot_tape.shape[0]
    t_setup = time.perf_counter() - t_setup
    episode_step = [0]
    last_outputs = [None]                  # (obs, agent_state, reward) of the latest step, device tensors

    def run_steps(n):
        """n x [step(actions_t); update()] as C calls over the device-resident tape (ants_rollout: no Python, no host
        round trip between the steps)."""
        done = 0
        while done < n:
            m = min(n_tape, n - done)
            last_outputs[0] = batch.rollout(rot_tape[:m], ph_tape[:m])
            done += m
        episode_step[0] += n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        run_steps(n)
        ev1.record()
        barrier()
        t = ev0.elapsed_time(ev1)
        if world > 1:
            tmax = torch.tensor([t], device="cuda", dtype=torch.float64)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            t = float(tmax.item())
        return t

    run_steps(W_)
    barrier()
    launches0 = batch.stats()["kernel_launches"]
    first_timed_step = episode_step[0]
    with ClockSampler(local_rank) as clocks:
        ms = timed(K)
    launches = batch.stats()["kernel_launches"] - launches0
    value = world * E * N * K / (ms / 1000.0)
    # the outputs of the last timed step, taken before the steps below overwrite them
    dumped = sample_outputs(*last_outputs[0]) if args.dump_outputs and rank == 0 else None

    # ---- per-kernel timing (the following K steps, CUDA events around every launch on the launching stream)
    batch.set_profiling(True)
    batch.reset_kernel_ms()
    barrier()
    run_steps(K)
    barrier()
    kms = batch.kernel_ms()
    st = batch.stats()
    batch.set_profiling(False)
    st["evap_mode"] = args.evap if gen.cfg["diffuse_factor"] == 0 else "dense"
    total_k = sum(v[0] for v in kms.values()) or 1.0
    kernels = {f: {"ms_per_step": v[0] / K, "launches_per_step": v[1] / K, "share": v[0] / total_k}
               for f, v in kms.items() if v[1]}
    dom = max(kernels, key=lambda f: kernels[f]["ms_per_step"])
    peak, peak_src = load_peaks()
    lps = max(kernels[dom]["launches_per_step"], 1e-9)
    dom_ms_per_launch = kernels[dom]["ms_per_step"] / lps
    abytes = algorithmic_bytes(dom, wl, E, C, st) / (lps if dom != "rocks" else 1.0)
    if dom == "rocks":
        dom_ms_per_launch = kernels[dom]["ms_per_step"]
    achieved = abytes / (dom_ms_per_launch / 1000.0) / 1e9
    traffic, traffic_src = ncu_traffic(dom, E * N)
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "dram_frac": (traffic / (dom_ms_per_launch / 1000.0) / 1e9 / peak) if traffic else None,
                "algorithmic_bytes_per_launch": abytes, "ms_per_launch": dom_ms_per_launch,
                "note": "frac: algorithmic bytes = SURVEY.md 8-d (the reference's f64 fields at element granularity, f32 obs) "
                        "/ event time / peak, i.e. how fast the reference's bytes are served (above 1 when the compact cell records carry them in fewer bytes than the survey counts); dram_frac: the DRAM bytes ncu "
                        "measured for this launch / event time / peak, i.e. how busy the HBM is (the 8-byte cell records "
                        "move far fewer bytes than the f64 planes)"}
    step_bytes = sum(algorithmic_bytes(f, wl, E, C, st) for f in kernels)
    roofline["step_achieved"] = step_bytes / (ms / K / 1000.0) / 1e9
    roofline["step_frac"] = roofline["step_achieved"] / peak
    roofline["bytes_per_ant_step"] = step_bytes / (E * N)

    # ---- the same K steps late in the episode (ants dispersed, long trails): untimed fast-forward, then timed
    late = None
    if late_start > 0:
        if episode_step[0] < late_start:
            run_steps(late_start - episode_step[0])
        late_first = episode_step[0]
        late_ms = timed(K)
        late = {"first_step": late_first, "steps": K, "ms_per_step": late_ms / K,
                "value": world * E * N * K / (late_ms / 1000.0), "vs_early": (late_ms / K) / (ms / K)}

    # ---- end to end through the host-buffer C ABI (numpy in, numpy out; copies inside the timed region)
    e2e, e2e_packed = None, None
    if args.e2e_steps > 0:
        h_rot = batch.pinned("rot", (E, N), np.int8)
        h_ph = batch.pinned("ph", (E, N), np.int8)
        h_rot[:] = rot_tape[0].cpu().numpy()
        h_ph[:] = ph_tape[0].cpu().numpy()
        L = batch.packed_layout()

        def time_e2e(step_fn):
            step_fn(h_rot, h_ph)
            batch.update_host(None)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            t0 = time.perf_counter()
            ev0.record()
            for _ in range(args.e2e_steps):
                step_fn(h_rot, h_ph)
                batch.update_host(None)
            ev1.record()
            barrier()
            e_ms = max(ev0.elapsed_time(ev1), (time.perf_counter() - t0) * 1000.0)
            if world > 1:
                tmax = torch.tensor([e_ms], device="cuda", dtype=torch.float64)
                dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                e_ms = float(tmax.item())
            return e_ms
        dense_bytes = E * N * (49 * C * 4 + 8 + 8)
        packed = bool(L.supported) and not os.environ.get("ANTS_E2E_DENSE") and E * N * 49 * C * 4 >= (4 << 20)
        pcie_bytes = E * N * (int(L.bytes_per_ant) + 8 + 8) if packed else dense_bytes
        e_ms = time_e2e(batch.step_host)
        pcie_peak = 56.3e9                     # pinned D2H copy measured on this pool (scripts/microbench/host_bw.cu)
        e2e = {"value": world * E * N * args.e2e_steps / (e_ms / 1000.0), "unit": "ant-steps/s",
               "h2d_bytes_per_step": 2 * E * N, "d2h_bytes_per_step": pcie_bytes, "host_result_bytes_per_step": dense_bytes,
               "steps": args.e2e_steps, "ms_per_step": e_ms / args.e2e_steps,
               "pcie_frac": pcie_bytes / (e_ms / args.e2e_steps / 1000.0) / pcie_peak,
               "host_write_gbs": dense_bytes / (e_ms / args.e2e_steps / 1000.0) / 1e9,
               "api": "ants_step_host + ants_update_host (pinned numpy buffers in, dense (E,N,7,7,C) f32 numpy out); "
                      + ("the observation crosses PCIe packed (visible samples, 12 B each) and is expanded to the dense array "
                         "by host threads inside the call" if packed else "dense device-to-host copy")}
        if packed:
            p_ms = time_e2e(batch.step_host_packed)
            e2e_packed = {"value": world * E * N * args.e2e_steps / (p_ms / 1000.0), "unit": "ant-steps/s",
                          "h2d_bytes_per_step": 2 * E * N, "d2h_bytes_per_step": pcie_bytes, "steps": args.e2e_steps,
                          "ms_per_step": p_ms / args.e2e_steps,
                          "pcie_frac": pcie_bytes / (p_ms / args.e2e_steps / 1000.0) / pcie_peak,
                          "api": "ants_step_host_packed + ants_update_host: the observation stays in its packed form on "
                                 "the host (ants_unpack_obs expands what the consumer needs)"}

    # ---- optional end-of-rollout statistics reduction (the only collective of the design)
    fin = batch.export_state(keys=("anthill_food", "holding"))
    local = torch.tensor([float(fin["anthill_food"].sum()), float(fin["holding"].sum())], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(local, op=dist.ReduceOp.SUM)
    rollout_stats = {"anthill_food_total": float(local[0].item()), "carried_food_total": float(local[1].item()),
                     "episode_steps": episode_step[0]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = run_cpu_baseline(wl, 3, args.cpu_steps)

    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)

    if rank == 0:
        line = {
            "metric": "ant-steps/sec (envs x ants x steps)", "value": value, "unit": "ant-steps/s",
            "n_gpus": world, "steps": K, "warmup": W_, "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s: %s" % (args.workload, wl["desc"]), "envs_per_gpu": E, "envs_total": E * world,
                       "ants_per_env": N, "map": [wl["w"], wl["h"]], "pheromones": wl["n_phero"], "rocks": wl["n_rocks"],
                       "obs": "7x7x%d f32" % C, "evaporation": st["evap_mode"], "cell_record": record,
                       "timed_steps": "steps %d-%d of the episode, one ants_rollout call" % (first_timed_step, first_timed_step + K),
                       "precision": "f64 positions / headings / sample coordinates; %s; f32 obs" % (
                           {"compact": "16 B cell records (f32 pheromone, bit-exact for saturated deposits via the decay "
                                       "table; f32 food)",
                            "compact8": "8 B cell records (u16 pheromone codes: saturated deposits bit-exact via the "
                                        "decay table, plain values in f32 side arrays; u16 food counts)"}.get(record, "f64 fields")), "l2": "state per GPU (%.1f GB) >> 126 MB L2"
                       % (st["device_bytes"] / 1e9), "parallelism": "env-sharded x%d, no per-step collective" % world,
                       "noise": "in-kernel Philox", "actions": "uniform random, pre-recorded tape on device"},
            "gpu_launches": int(launches), "clocks": clocks.summary(), "roofline": roofline, "kernels": kernels,
            "late": late, "e2e": e2e, "e2e_packed": e2e_packed, "cpu_baseline": cpu, "rollout_stats": rollout_stats,
            "setup_s": t_setup,
        }
        emit(line)
    batch.close()
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """The reference's own CPU implementation of the path: the UNMODIFIED reference (oracle/_ref, byte-compiled from
    /root/reference by oracle/build_ref.py; the oracle port only if that is missing), all host cores, one env per
    process; each bench step = one step()+update() of every env."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    procs = os.cpu_count() or 1
    r = run_cpu_baseline(wl, max(args.warmup, 3), args.steps, procs)
    line = {"impl": "reference", "metric": "ant-steps/sec (envs x ants x steps)", "value": r["value"],
            "unit": "ant-steps/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_env_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s: %s" % (args.workload, wl["desc"]), "envs_total": procs,
                       "ants_per_env": wl["n_ants"], "map": [wl["w"], wl["h"]]},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "ant-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ----------------------------------------------------------------------------------------------- configs[0]: the drop-in
DROPIN_LOOP = """
import sys, types, json, time
for name in ("noise", "matplotlib", "matplotlib.pyplot"):
    sys.modules.setdefault(name, types.ModuleType(name))
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
ROOT, REF, USE_DROPIN, K, W = %(root)r, %(ref)r, %(dropin)r, %(k)d, %(w)d
if USE_DROPIN:
    sys.path.insert(0, ROOT)
    import antsrl_b200
    sys.path.insert(0, antsrl_b200.dropin_path())
else:
    sys.path.insert(0, REF)
import numpy as np
from environment.RL_api import RLApi
from environment.rewards.reward_custom import All_Rewards
from generator.environment_generator import EnvironmentGenerator
from generator.map_generators import CirclesGenerator
api = RLApi(All_Rewards(1, 2, 10, 1, 3), 1, 1, 40 / 180 * np.pi, 0.05, 0.5)               # main.py:42-50
gen = EnvironmentGenerator(200, 200, 50, 2, 0, CirclesGenerator(20, 5, 10), CirclesGenerator(10, 5, 15), K + W + 1, seed=1000)
env = gen.generate(api)                                                                  # main.py:79
api.ants.activate_all_pheromones(np.ones((50, 2)) * 10)                                  # agent.initialize
np.random.seed(777)
act = np.random.RandomState(4242)
obs, agent_state, state = api.observation()                                              # main.py:88
t0 = None
for s in range(W + K):
    if s == W:
        t0 = time.perf_counter()
    rot = act.randint(0, 3, 50) - 1                                                      # the agents' exploration branch
    ph = act.randint(0, 3, 50)
    obs, agent_state, reward, done = api.step(rot, ph)                                   # main.py:98
    env.update()                                                                         # main.py:131
dt = time.perf_counter() - t0
print(json.dumps({"ms_per_step": dt * 1000 / K, "reward_sum": float(np.sum(reward)), "obs_shape": list(obs.shape)}))
"""


def run_dropin(args):
    """BASELINE.json configs[0]: the reference's default generated map (200x200, 50 ants) driven for K steps by random
    actions through main.py's loop -- once over the drop-in packages (environment / generator of antsrl_b200.dropin: ONE
    environment per handle, numpy in / numpy out, the reference's global-RNG collision noise) and once over the
    unmodified reference on the host."""
    from oracle import ref_harness
    K, W_ = args.steps, max(args.warmup, 3)
    out = {}
    for name, use in (("dropin", True), ("reference", False)):
        if not use and not ref_harness.reference_available():
            continue
        code = DROPIN_LOOP % dict(root=ROOT, ref=ref_harness.REFERENCE_ROOT, dropin=use, k=K, w=W_)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=3000)
        if r.returncode != 0:
            sys.stderr.write(r.stderr[-3000:])
            raise SystemExit("bench.py: the %s loop failed" % name)
        out[name] = json.loads(r.stdout.strip().splitlines()[-1])
    d = out["dropin"]
    line = {"metric": "ant-steps/sec (envs x ants x steps)", "value": 50 * 1000.0 / d["ms_per_step"], "unit": "ant-steps/s",
            "n_gpus": 1, "steps": K, "warmup": W_, "ms_per_step": d["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "cfg1: reference default generated map 200x200, 50 ants, ONE environment through the drop-in "
                                   "RLApi / Environment classes (main.py's loop, random actions, reference's global-RNG noise)"},
            "reference_ms_per_step": out.get("reference", {}).get("ms_per_step"),
            "speedup_vs_reference": (out["reference"]["ms_per_step"] / d["ms_per_step"]) if "reference" in out else None,
            "note": "one small environment per call is latency bound (launches + the host round trip of every call); the "
                    "batched path (default workload) is the throughput configuration"}
    emit(line)


def torchrun_command(n_gpus, argv, port=None):
    """The contract's multi-GPU launch of this script: one process per GPU on one node, rendezvous on 127.0.0.1."""
    port = port or (29500 + os.getpid() % 2000)
    return [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(int(n_gpus)),
            "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + list(argv)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def make_parser():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS) + ["cfg1"],
                    help="cfg1 = BASELINE configs[0]: ONE default environment through the drop-in classes")
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the workload's)")
    ap.add_argument("--evap", default="lazy", choices=["lazy", "tiles", "dense"])
    ap.add_argument("--record", default="compact8", choices=["compact8", "compact", "f64"],
                    help="cell record format (compact8 = 8 B, compact = 16 B: lazy mode only)")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--cpu-steps", type=int, default=40)
    ap.add_argument("--late-start", type=int, default=900,
                    help="episode step at which the K steps are timed again (0 = skip the late window)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them returned (obs, agent_state, reward; rank "
                         "0's envs) as DIR/<name>.npy, at most 64 MB: a fixed sample of the ants when all do not fit")
    return ap


def main():
    # Libraries print on fd 1 (NCCL's version banner comes from C, whatever NCCL_DEBUG says): everything but the
    # final JSON line is sent to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = make_parser()
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload == "cfg1"):
        ap.error("--dump-outputs writes the outputs of the GPU step loop (--impl ours, workload cfg2/cfg3/cfg4)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "ours" and args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # `python bench.py --gpus N` typed by hand: become the launch the driver uses (one rank per GPU over NCCL)
        os.dup2(_REAL_STDOUT, 1)
        cmd = torchrun_command(args.gpus, sys.argv[1:])
        os.execv(cmd[0], cmd)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "ours" and args.gpus != world:
        sys.stderr.write("bench.py: --gpus %d but WORLD_SIZE=%d; running on %d rank(s)\n" % (args.gpus, world, world))
    if args.workload == "cfg1":
        run_dropin(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
