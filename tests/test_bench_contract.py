"""bench.py prints ONE JSON line with the keys the driver reads (metric / value / roofline /
cpu_baseline / e2e / gpu_launches / clocks); checked on CPU for the reference arm and on a B200 for
the GPU arm at a reduced env count."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def run_bench(*flags, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def check_reference_line(d, kind):
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        baseline = json.load(f)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == baseline["metric"] and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "experiment 6" in d["config"]["workload"] and d["gpu_launches"] == 0
    ran = d["config"]["reference_arm_ran"]          # the config says what this arm really ran (a bounded sample)
    assert ran["experiment"] == 6 and ran["envs"] >= 1


def test_reference_arm_line_port():
    """--impl reference --ref-port: the C restatement of the reference algorithm on the host cores (the fallback
    when the staged reference is missing)."""
    d = run_bench("--impl", "reference", "--steps", "2", "--warmup", "3", "--ref-budget-s", "4", "--ref-port")
    check_reference_line(d, "port")
    assert d["value"] > 1e5 and "C port" in d["config"]["reference_arm_ran"]["implementation"]


def test_reference_arm_line_real_reference():
    """--impl reference: the UNMODIFIED reference BoatEnv, one process per core (oracle/_ref or /root/reference)."""
    sys.path.insert(0, ROOT)
    from oracle import ref_shim
    if not ref_shim.reference_available():
        pytest.skip("reference neither mounted nor staged (python oracle/make_ref.py)")
    d = run_bench("--impl", "reference", "--steps", "2", "--warmup", "3", "--ref-budget-s", "6")
    check_reference_line(d, "reference")
    ran = d["config"]["reference_arm_ran"]
    assert ran["processes"] == d["cpu_baseline"]["cores"] and "unmodified" in ran["implementation"]
    assert 1e3 < d["value"] < 1e7                     # ~1e4 env-steps/s per core (SURVEY.md section 6)


def test_make_ref_stages_byte_identical_copies(tmp_path):
    """oracle/make_ref.py: the staged files are the reference's own bytes, and the shim imports from the copy."""
    sys.path.insert(0, ROOT)
    from oracle import make_ref
    if not os.path.isfile(os.path.join(make_ref.DEFAULT_SRC, "environment", "boat_env.py")):
        pytest.skip("reference not mounted")
    dest = make_ref.make_ref(dest=str(tmp_path / "_ref"))
    assert make_ref.check(dest)
    for rel in make_ref.HOT_PATH:
        with open(os.path.join(make_ref.DEFAULT_SRC, rel), "rb") as a, open(os.path.join(dest, rel), "rb") as b:
            assert a.read() == b.read(), rel
    code = ("import sys; sys.path.insert(0, %r); from oracle import ref_shim as R; import numpy as np; np.random.seed(0); "
            "env = R.make_env(R.load_config(base_settings__experiment=6)); o = env.reset(); "
            "o, r, d, i = env.step(np.array([0.5], dtype=np.float32)); print(R.REFERENCE_ROOT, float(o[1]))" % ROOT)
    env = dict(os.environ, SAC_REFERENCE_ROOT=dest)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    root, vx = r.stdout.split()
    assert root == dest and float(vx) == 3.0 / 5.0     # step 1 sets v_x = 3 (control_blocks.py:21-22), obs = v_x / 5


@pytest.mark.gpu
def test_gpu_arm_line():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    n = 1 << 20
    d = run_bench("--steps", "20", "--warmup", "30", "--envs-per-gpu", str(n), "--e2e-steps", "3", "--no-cpu-baseline",
                  "--no-toys")
    assert (BASE_KEYS - {"cpu_baseline"}) <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["dtype"] == "f32" and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["value"] > 1e9 and d["ms_per_step"] > 0
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and 0 < rf["frac"] < 1.2
    assert rf["achieved"] == pytest.approx(165 * n / (rf["kernel_ms"] * 1e-3) / 1e9, rel=1e-6)
    assert d["e2e"]["h2d_bytes_per_step"] == 4 * n and d["e2e"]["d2h_bytes_per_step"] == (44 + 4 + 1) * n
    assert 0 < d["e2e"]["value"] < d["value"]
    assert d["gpu_launches"] >= 2 * 20          # one policy launch + one step launch per step
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    # the timed region is in the steady-state reset regime whatever --warmup is, and contains a statistics all-reduce
    assert d["config"]["preroll_steps"] >= 400 and d["stats_allreduces_in_timed_region"] >= 1
    assert d["episodes_finished_in_timed_region"] > 0.5 * 20 * n / 362
    k = d["e2e_k"]
    assert k["substeps_per_call"] == 8 and k["h2d_bytes_per_step"] == 8 * 4 * n and k["value"] > d["e2e"]["value"]


@pytest.mark.gpu
def test_gpu_arm_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs: the last timed step's outputs for a fixed env sample, identical from run to run, with
    --steps timed steps (one policy launch + one step launch each)."""
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    n, steps = 1 << 19, 7
    flags = ["--steps", str(steps), "--warmup", "3", "--envs-per-gpu", str(n), "--e2e-steps", "3", "--e2e-k", "0",
             "--no-cpu-baseline", "--no-toys"]
    runs = []
    for i in range(2):
        d = run_bench(*flags, "--dump-outputs", str(tmp_path / str(i)))
        assert d["steps"] == steps and 2 * steps <= d["gpu_launches"] <= 2 * steps + 4
        runs.append({f[:-4]: np.load(tmp_path / str(i) / f) for f in sorted(os.listdir(tmp_path / str(i)))})
    a, b = runs
    m = 1 << 18
    assert sorted(a) == ["action", "done", "env_index", "final_obs", "obs", "reward", "term"]
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert a["obs"].shape == a["final_obs"].shape == (m, 11) and a["reward"].shape == a["done"].shape == (m,)
    idx = a["env_index"]
    assert len(np.unique(idx)) == m and idx.min() >= 0 and idx.max() < n and np.all(idx == np.floor(idx))
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert np.isfinite(a["obs"]).all() and np.array_equal(a["done"], (a["term"] != 0).astype(np.float32))
    # the dumped actions are the policy's draw for the last timed step (after pre-roll and warm-up) at the sampled ids
    import bench
    import sac_agent_b200 as S
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=bench.EXPERIMENT), n, seed=bench.SEED,
                           precision="fp32", device=0)
    rows = idx.astype(np.int64)
    last = bench.PREROLL + 3 + steps - 1
    assert np.array_equal(a["action"], env.uniform_actions(last).cpu().numpy()[rows])
    assert not np.array_equal(a["action"], env.uniform_actions(last - 1).cpu().numpy()[rows])
    env.close()


@pytest.mark.gpu
def test_gpu_arm_strong_scaling_line():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    d = run_bench("--steps", "10", "--warmup", "5", "--scaling", "strong", "--total-envs", str(1 << 21), "--e2e-steps", "3",
                  "--no-cpu-baseline", "--no-toys", "--e2e-k", "0")
    assert d["scaling"] == "strong" and d["config"]["total_envs"] == 1 << 21 and d["config"]["envs_per_gpu"] == 1 << 21
    assert d["value"] > 1e9 and d["e2e_k"] is None
