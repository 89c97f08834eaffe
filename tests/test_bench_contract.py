"""bench.py's contract, as far as it can be checked without a GPU: the reference arm (`--impl reference`, the
reference algorithm on the host cores) prints ONE JSON line with the contract's keys, ranks other than 0 stay silent,
and the algorithmic-byte accounting matches SURVEY.md section 8-d / DESIGN.md section 3.  On a GPU: `--dump-outputs`
writes the same outputs in two runs with the same arguments."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, *flags):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg2",
                        "--steps", "3", "--warmup", "1", *flags], capture_output=True, text=True, cwd=ROOT, env=env,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout


def test_reference_arm_prints_one_contract_line():
    out = _run()
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "ant-steps/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("ant-steps/sec") and d["steps"] == 3 and d["warmup"] == 3 and d["value"] > 0   # W >= 3
    assert d["config"]["workload"].startswith("cfg2") and d["data"] == "synthetic" and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    sys.path.insert(0, ROOT)
    from oracle import ref_harness
    # the unmodified reference (checkout, or oracle/_ref built by oracle/build_ref.py) wherever it exists
    assert cb["kind"] == ("reference" if ref_harness.reference_available() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "ant-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    out = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, "--gpus", "2")
    assert out.strip() == ""


def test_algorithmic_bytes_follow_the_survey():
    sys.path.insert(0, ROOT)
    import bench
    wl = bench.WORKLOADS["cfg4"]
    E, N, P = 512, wl["n_ants"], wl["n_phero"]
    # perception: obs f32 + agent_state + reward out, 49 samples x (phero, food, walls, explored r/w), per-ant state
    per_ant = 49 * 7 * 4 + 16 + 49 * (8 * P + 8 + 3) + 82
    assert per_ant == 2793                                                   # DESIGN.md section 3
    assert bench.algorithmic_bytes("perceive", wl, E, 7, {}) == E * N * per_ant
    assert bench.algorithmic_bytes("perceive", bench.WORKLOADS["cfg3"], 1, 6, {}) == 256 * 2597
    assert bench.algorithmic_bytes("evaporate", wl, E, 7, {"evap_mode": "lazy"}) == 0
    assert bench.algorithmic_bytes("evaporate", wl, E, 7, {"evap_mode": "dense"}) == E * 1024 * 1024 * (16 * P + 1)
    step = sum(bench.algorithmic_bytes(f, wl, E, 7, {"evap_mode": "lazy"})
               for f in ("move", "perceive", "collide", "rocks", "deposit")) / (E * N)
    assert abs(step - 3109) < 1                                              # bytes per ant-step in the bench line
    # the block-per-environment kernels carry the algorithmic bytes of the flat kernels they replace
    fused = sum(bench.algorithmic_bytes(f, wl, E, 7, {"evap_mode": "lazy"}) for f in ("perceive", "env_update_move")) / (E * N)
    assert abs(fused - step) < 1e-9
    peak, src = bench.load_peaks()
    assert 5000 < peak < 9000 and ("measured" in src or "fallback" in src)


def test_dump_outputs_sample_is_fixed_and_bounded(monkeypatch):
    """--dump-outputs: every ant while they fit, else the documented seeded sample of rows, the same rows in every array;
    obs / agent_state stay f32 and reward f64."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    rs = np.random.RandomState(1)
    E, N, S, C = 3, 40, 7, 6
    obs = torch.from_numpy(rs.random_sample((E, N, S, S, C)).astype(np.float32))
    ast = torch.from_numpy(rs.random_sample((E, N, 2)).astype(np.float32))
    rew = torch.from_numpy(rs.random_sample((E, N)))
    full = bench.sample_outputs(obs, ast, rew)
    assert np.array_equal(full["obs"], obs.numpy().reshape(E * N, S, S, C))
    assert np.array_equal(full["agent_state"], ast.numpy().reshape(E * N, 2))
    assert np.array_equal(full["reward"], rew.numpy().reshape(E * N))
    per_ant = S * S * C * 4 + 2 * 4 + 8
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 4096 + 50 * per_ant)
    part = bench.sample_outputs(obs, ast, rew)
    rows = np.sort(np.random.RandomState(0).choice(E * N, 50, replace=False))
    assert part["obs"].dtype == np.float32 and part["agent_state"].dtype == np.float32 and part["reward"].dtype == np.float64
    assert np.array_equal(part["obs"], full["obs"][rows]) and np.array_equal(part["agent_state"], full["agent_state"][rows])
    assert np.array_equal(part["reward"], full["reward"][rows])
    assert sum(a.nbytes for a in part.values()) <= bench.DUMP_BYTES


def test_dump_outputs_is_refused_where_there_is_no_gpu_step_loop():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and r.stdout == ""


@pytest.mark.gpu
def test_dump_outputs_are_those_of_the_last_timed_step(tmp_path):
    """Two runs with the same arguments time exactly --steps steps and write the same outputs; they are the outputs of
    the last timed step: the same inputs driven here through the warm-up and timed rollouts give them again."""
    import numpy as np
    args = ["--workload", "cfg2", "--envs", "16", "--steps", "7", "--warmup", "3", "--late-start", "0", "--e2e-steps", "0",
            "--no-cpu-baseline"]
    for k in range(2):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / str(k))],
                           capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout)
        assert d["steps"] == 7 and d["config"]["timed_steps"].startswith("steps 3-10 ")
    names = ("agent_state", "obs", "reward")
    assert sorted(os.listdir(tmp_path / "0")) == [n + ".npy" for n in names]
    got = [{n: np.load(str(tmp_path / str(k) / (n + ".npy"))) for n in names} for k in range(2)]
    assert got[0]["obs"].shape == (16 * 50, 7, 7, 6) and got[0]["obs"].dtype == np.float32
    assert got[0]["agent_state"].shape == (16 * 50, 2) and got[0]["reward"].shape == (16 * 50,)
    assert got[0]["reward"].dtype == np.float64 and np.abs(got[0]["obs"]).sum() > 0
    for n in names:
        assert np.array_equal(got[0][n], got[1][n]), n
    sys.path.insert(0, ROOT)
    import bench
    a = bench.make_parser().parse_args(args)
    _, batch, _, rot, ph = bench.make_batch(a)
    try:
        batch.rollout(rot[:a.warmup], ph[:a.warmup])
        want = bench.sample_outputs(*batch.rollout(rot[:a.steps], ph[:a.steps]))
    finally:
        batch.close()
    for n in names:
        assert np.array_equal(got[0][n], want[n]), n


def test_hand_typed_multi_gpu_run_becomes_the_torchrun_launch():
    sys.path.insert(0, ROOT)
    import bench
    cmd = bench.torchrun_command(4, ["--gpus", "4", "--steps", "50"], port=29777)
    assert cmd[:3] == [sys.executable, "-m", "torch.distributed.run"]
    assert cmd[3:10] == ["--nnodes=1", "--nproc-per-node", "4", "--master-addr", "127.0.0.1", "--master-port", "29777"]
    assert cmd[10] == os.path.join(ROOT, "bench.py") and cmd[11:] == ["--gpus", "4", "--steps", "50"]
