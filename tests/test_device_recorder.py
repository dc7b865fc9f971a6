"""DeviceRecorder: the reference's recorder CSVs (postprocessing/recorder.py:18-56) recorded on the device.

CPU tests: the bookkeeping shared by both recorders against hand-written CSV text, and the record kernel's
register budget.  GPU tests: byte equality with BatchedRecorder (plain step and the fused step + store, fp32 and
fp64, automatic flushes mid-run), the recorded fixture-6 episode, ring contents at benchmark size, shard naming and
id checks, and examples/train_sac.py --record-envs with and without --overlap.
"""
import importlib.util
import os
import re
import subprocess

import numpy as np
import pytest

from boat_testlib import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("s_x", "s_y", "v_x", "v_y", "s_r", "rudder_angle")


@pytest.fixture(scope="module")
def S():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import sac_agent_b200 as pkg
    pkg.lib()  # raises if libboatenv.so is missing: the GPU tests never run on a fallback
    return pkg


def tree(path):
    """{relative path: bytes} of every file under path."""
    out = {}
    for d, _, files in os.walk(path):
        for f in files:
            p = os.path.join(d, f)
            out[os.path.relpath(p, path)] = open(p, "rb").read()
    return out


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
def test_episode_book_rows_and_naming(tmp_path):
    """Two envs, the second one terminating in the middle: zeroed action / reward on the first row of the next
    episode, cumulative info counters, one data file per episode, ``env<id>_`` prefixes."""
    from sac_agent_b200.csv_export import DATA_COLUMNS, INFO_COLUMNS, EpisodeBook, _append_rows
    f = np.float64
    book = EpisodeBook([3, 7], str(tmp_path))

    def write(rows):
        for path, row in rows:
            _append_rows(path, DATA_COLUMNS, [row])

    write([book.data_row(3, f(1.5), f(-2.0), f(0.0), f(0.25), f(0.5), f(0.0)),
           book.data_row(7, f(2.5), f(1.0), f(0.0), f(0.0), f(0.0), f(0.125))])
    assert book.after_step(3, f(0.5), f(1.25), np.uint8(0)) is None
    path, row = book.after_step(7, f(-0.75), f(-0.5), np.uint8(5))        # rudder_broken
    _append_rows(path, INFO_COLUMNS, [row])
    write([book.data_row(3, f(1.75), f(-2.0), f(0.5), f(0.25), f(0.5), f(0.0625)),
           book.data_row(7, f(0.0), f(3.0), f(0.0), f(0.0), f(0.0), f(0.0))])
    assert book.after_step(3, f(0.25), f(0.75), np.uint8(0)) is None
    path, row = book.after_step(7, f(1.0), f(2.0), np.uint8(1))           # reached_goal
    _append_rows(path, INFO_COLUMNS, [row])
    header = ";".join(DATA_COLUMNS) + "\r\n"
    ep = tmp_path / "episodes"
    assert sorted(os.listdir(ep)) == ["env3_episode_0_data.csv", "env7_episode_0_data.csv",
                                      "env7_episode_1_data.csv", "env7_info.csv"]
    assert (ep / "env3_episode_0_data.csv").read_bytes().decode() == header + (
        "1.5;-2.0;0.0;0.25;0.5;0;0;0.0;20\r\n"
        "1.75;-2.0;0.5;0.25;0.5;0.5;1.25;0.0625;20\r\n")
    assert (ep / "env7_episode_0_data.csv").read_bytes().decode() == header + "2.5;1.0;0.0;0.0;0.0;0;0;0.125;20\r\n"
    assert (ep / "env7_episode_1_data.csv").read_bytes().decode() == header + "0.0;3.0;0.0;0.0;0.0;0;0;0.0;20\r\n"
    assert (ep / "env7_info.csv").read_bytes().decode() == (
        "termination;reached_goal;out_of_bounds;out_of_fuel;rudder_broken;timeout;episode_reward\r\n"
        "rudder_broken;0;0;0;1;0;-0.5\r\n"
        "reached_goal;1;0;0;1;0;2.0\r\n")
    assert book.info[3]["episode_reward"] == 2.0 and book.episode == {3: 0, 7: 2}
    # the naming rule: no prefix only when the sole recorded id is 0
    assert os.path.basename(EpisodeBook([0], str(tmp_path)).name(0, "info.csv")) == "info.csv"
    assert os.path.basename(EpisodeBook([0, 1], str(tmp_path)).name(0, "info.csv")) == "env0_info.csv"
    assert os.path.basename(EpisodeBook([5], str(tmp_path)).name(5, "wind.csv")) == "env5_wind.csv"


def test_record_kernel_compiles_without_spills(tmp_path):
    from sac_agent_b200 import _build
    src = os.path.join(_build.CSRC, "record.cu")
    r = subprocess.run([_build.nvcc(), "-Xptxas=-v", *_build.ARCH, *_build.COMMON, "-c", src, "-o",
                        str(tmp_path / "record.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    blocks = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads", r.stderr)
    record = [b for b in blocks if "boat_record_kernel" in b[0]]
    assert len(record) == 2, r.stderr   # float and double
    assert all(b[1:] == ("0", "0", "0") for b in record), record


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("fused", [False, True], ids=["step", "step_store"])
def test_device_recorder_matches_batched_recorder(S, tmp_path, precision, fused):
    """4099 envs (a ragged last tile block), experiment 6, actions of scale 2: several rudder_broken episodes per
    env under auto-reset.  A 256-row ring flushes itself four times over the 1200 steps.  Both trees are equal
    byte for byte."""
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), 4099, seed=3, precision=precision, device=0)
    mem = S.ReplayBuffer(8192, (11,), 1, precision=precision, device=0) if fused else None
    ids = [0, 31, 32, 1000, 4098] + [int(i) for i in np.random.default_rng(7).choice(np.arange(33, 4098), 4, False)]
    env.reset()
    host = S.BatchedRecorder(env, ids, str(tmp_path / "host"))
    host.write_winds_to_csv()
    dev = S.DeviceRecorder(env, ids, str(tmp_path / "device"), capacity=256)
    dev.start()
    for t in range(1200):
        a = env.uniform_actions(t, 2.0)
        host.write_data_to_csv()
        if fused:
            mem.step_store(env, a)
        else:
            env.step(a)
        host.after_step(a)
        dev.capture(a)
    host.write_data_to_csv()
    dev.close()
    a, b = tree(tmp_path / "host"), tree(tmp_path / "device")
    assert sorted(a) == sorted(b)
    assert all(a[k] == b[k] for k in a), [k for k in a if a[k] != b[k]][:5]
    assert min(host.episode.values()) >= 1 and dev.episodes_finished == sum(host.episode.values())
    env.close()
    if mem:
        mem.close()


@pytest.mark.gpu
def test_device_recorder_reproduces_fixture_6(S, tmp_path):
    """The recorded fixture-6 episode (test_mode 1) through both recorders: identical files, so the device path
    reproduces the reference's episode_0_data.csv / wind.csv / info.csv exactly as BatchedRecorder does."""
    import pandas as pd
    import torch
    g = load_golden("fixture_exp6")
    fp = int(g["config"]["wind"]["fixed_points"])
    knots = np.zeros((1, 2, fp))
    knots[0, 0], knots[0, 1] = g["knots_v"], g["knots_a"]
    env = S.BatchedBoatEnv(g["config"], 1, precision="fp64", device=0, auto_reset=True)
    env.set_episode_draws(np.array([0]), knots)
    env.reset()
    host = S.BatchedRecorder(env, [0], str(tmp_path / "host"))
    host.write_winds_to_csv()
    dev = S.DeviceRecorder(env, [0], str(tmp_path / "device"), capacity=1024)
    dev.start()
    zero = torch.zeros(1, dtype=env.dtype, device=env.device)
    done = False
    while not done:
        host.write_data_to_csv()
        _, _, d, _ = env.step(zero)
        host.after_step(zero)
        dev.capture(zero)
        done = bool(d[0])
    host.write_data_to_csv()
    dev.close()
    a, b = tree(tmp_path / "host"), tree(tmp_path / "device")
    assert sorted(a) == sorted(b) and all(a[k] == b[k] for k in a)
    data = pd.read_csv(tmp_path / "device" / "episodes" / "episode_0_data.csv", sep=";")
    assert len(data) == int(g["n_rows"])
    info = pd.read_csv(tmp_path / "device" / "episodes" / "info.csv", sep=";")
    assert info.termination[0] == "reached_goal"
    assert info.episode_reward[0] == pytest.approx(871.2727580297085, abs=1e-8)
    env.close()


@pytest.mark.gpu
def test_ring_equals_get_field_at_benchmark_size(S, tmp_path):
    """16,777,235 envs (fp32, experiment 6), 64 recorded ids from the first block, blocks far into the sweep and
    the ragged tail.  Before every flush, each ring row is bitwise what get_field / reward / term / episode gave
    for the step it belongs to."""
    import torch
    n = 16_777_235
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), n, seed=11, precision="fp32", device=0)
    fixed = list(range(8)) + [31, 32, 33, 8_388_607, 8_388_608, n - 20, n - 19, n - 3, n - 1]   # n - 19: last block
    rand = [int(x) for x in np.random.default_rng(5).choice(np.arange(64, n - 64), 64, replace=False)]
    ids = list(dict.fromkeys(fixed + rand))[:64]
    idx = torch.tensor(ids, dtype=torch.int64, device=env.device)
    env.reset()
    cap = 128
    rec = S.DeviceRecorder(env, ids, str(tmp_path), capacity=cap)

    def expected(a=None):
        cols = {f: env.get_field(f)[idx] for f in FIELDS}
        cols["episode"] = env.get_field("episode")[idx]
        z = torch.zeros(len(ids), dtype=env.dtype, device=env.device)
        cols["action"] = a[idx] if a is not None else z
        cols["reward"] = env.reward[idx].clone() if a is not None else z
        cols["term"] = env.term[idx].clone() if a is not None else torch.zeros(len(ids), dtype=torch.uint8,
                                                                              device=env.device)
        return cols

    def bits(t):
        return t.view(torch.int32) if t.dtype == torch.float32 else t

    want = [expected()]
    rec.start()
    checked = 0
    for t in range(400):
        a = env.uniform_actions(t, 2.0)
        env.step(a)
        rec.capture(a)
        want.append(expected(a))
        if rec.pending == cap or t == 399:
            torch.cuda.synchronize()
            for r, w in enumerate(want):
                slot = (rec._flushed + r) % cap
                for k, v in w.items():
                    assert torch.equal(bits(rec._cols[k][slot]), bits(v)), (t, r, k)
                checked += 1
            rec.flush()
            want = []
    assert checked == 401
    rec.close()
    env.close()


@pytest.mark.gpu
def test_shard_ids_and_errors(S, tmp_path):
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), 100, seed=2, precision="fp32", device=0,
                           env_id_offset=5000)
    env.reset()
    s_x0 = float(env.get_field("s_x")[42])
    for bad in ([4999], [5100], [5001, 5001], []):
        with pytest.raises(ValueError):
            S.DeviceRecorder(env, bad, str(tmp_path))
    rec = S.DeviceRecorder(env, [5000, 5042, 5099], str(tmp_path), capacity=8)
    rec.start()
    for t in range(20):
        a = env.uniform_actions(t, 0.5)
        env.step(a)
        rec.capture(a)
    rec.close()
    names = sorted(os.listdir(tmp_path / "episodes"))
    for g in (5000, 5042, 5099):
        assert f"env{g}_episode_0_data.csv" in names and f"env{g}_wind.csv" in names
    assert {int(re.match(r"env(\d+)_", x).group(1)) for x in names} == {5000, 5042, 5099}
    # the first row is the state after reset of the shard's local env 42
    first = open(tmp_path / "episodes" / "env5042_episode_0_data.csv").read().splitlines()[1].split(";")
    assert float(first[0]) == s_x0
    env.close()


def _train_sac():
    spec = importlib.util.spec_from_file_location("train_sac", os.path.join(ROOT, "examples", "train_sac.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, True], ids=["sequential", "overlap"])
def test_train_sac_records_envs(S, tmp_path, overlap):
    import pandas as pd
    from sac_agent_b200.csv_export import DATA_COLUMNS
    args = ["--envs", "4096", "--iters", "300", "--buffer", "65536", "--experiments-root", str(tmp_path / "rec"),
            "--record-envs", "4", "--log-every", "50"] + (["--overlap"] if overlap else [])
    out = _train_sac().main(args)
    ep = os.path.join(out["experiment_dir"], "episodes")
    names = os.listdir(ep)
    assert out["recorded_envs"] == 4
    n_info = 0
    for g in range(4):
        data = [x for x in names if re.fullmatch(rf"env{g}_episode_\d+_data\.csv", x)]
        assert f"env{g}_wind.csv" in names
        rows = 0
        for x in data:
            df = pd.read_csv(os.path.join(ep, x), sep=";")
            assert tuple(df.columns) == DATA_COLUMNS and (df.n == 20).all()
            rows += len(df)
        assert rows == 20 + 300 + 1     # warm-up and timed iterations, plus the state after reset
        info = pd.read_csv(os.path.join(ep, f"env{g}_info.csv"), sep=";") if f"env{g}_info.csv" in names else None
        k = 0 if info is None else len(info)
        if info is not None:
            assert set(info.termination) <= set(S.TERM_NAMES[1:])
        assert len(data) == k + 1
        n_info += k
    assert out["recorded_episodes"] == n_info
    assert not any(x.startswith("env4_") for x in names)
    plain = _train_sac().main(["--envs", "4096", "--iters", "20", "--warmup-iters", "0", "--buffer", "65536",
                               "--experiments-root", str(tmp_path / "plain"), "--log-every", "10"]
                              + (["--overlap"] if overlap else []))
    assert os.listdir(os.path.join(plain["experiment_dir"], "episodes")) == []
    assert "recorded_envs" not in plain
