"""Experiment-directory compatibility (SURVEY.md 8f rank 3): tree, tuned-config draw and summary CSVs in
the formats of utils/build_experiment.py:9-41, utils/hyperparameter_tuner.py:9-52 and main.py:116-133.
The expected headers are those of the reference's own recorded experiments
(ressources/settings_visualized/experiment_setting_1/{console,terminations}.csv)."""
import csv
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sac_agent_b200 as S  # noqa: E402


def test_experiment_tree_configs_and_csvs(tmp_path):
    exp = S.Experiment(subdir="setting_5", root=str(tmp_path), rng=random.Random(3))
    assert exp.experiment_name.startswith("experiment_") and os.path.isdir(exp.experiment_dir)
    assert exp.experiments_dir == os.path.join(str(tmp_path), "setting_5")
    for d in ("plots", "checkpoints", "configs", "rendering", "episodes"):
        assert os.path.isdir(os.path.join(exp.experiment_dir, d))
    cfg = S.load_config(base_settings__experiment=5)
    tuned = exp.save_configs(cfg)
    orig = S.get_experiment_config(exp.experiment_dir, "original_config.yaml")
    assert orig.agent.learning_rate_alpha == 0.005 and orig.boat.fuel == 15000
    h = exp.tuner.hpset
    assert tuned.agent.learning_rate_alpha == h["alpha"] and tuned.agent.tvn_parameter_modulation_tau == h["tau"]
    assert 0.001 <= h["alpha"] <= 0.01 and 0.0008 <= h["beta"] <= 0.008 and 0.95 <= h["gamma"] <= 0.99
    assert all(round(v, 4) == v for v in h.values())
    assert tuned.boat == orig.boat and tuned.wind == orig.wind        # only the four agent keys change
    assert S.params_from_config(tuned).fuel == 15000.0                # a tuned config drives the env unchanged
    # same seed, same draw; another seed, another member
    assert S.HPTuner(rng=random.Random(3)).hpset == h and S.HPTuner(rng=random.Random(4)).hpset != h

    counters = {"reached_goal": 2, "out_of_bounds": 5, "out_of_fuel": 0, "timeout": 1, "rudder_broken": 40,
                "episodes": 48.0, "return_sum": -4800.0, "return_sumsq": 1e6}
    info = S.info_from_counters(counters, "rudder_broken")
    exp.write_console([[(0, 50), "rudder_broken-40", -101.5, -99.0, -100.0, "", ""]])
    exp.append_overview(-99.0)
    exp.append_overview(-98.0)
    exp.write_terminations(info)
    rows = list(csv.reader(open(os.path.join(exp.experiment_dir, "console.csv")), delimiter=";"))
    assert rows[0] == ["CCID Episode", "Termination", "Score", "Best Score", "Average Score", "RA", "Action RA"]
    assert rows[1][:3] == ["(0, 50)", "rudder_broken-40", "-101.5"]
    rows = list(csv.reader(open(os.path.join(exp.experiment_dir, "terminations.csv")), delimiter=";"))
    assert rows[0] == ["termination", "reached_goal", "out_of_bounds", "out_of_fuel", "rudder_broken", "timeout",
                       "episode_reward"]
    assert rows[1] == ["rudder_broken", "2", "5", "0", "40", "1", "-100.0"]
    rows = list(csv.reader(open(os.path.join(exp.experiments_dir, "overview.csv")), delimiter=";"))
    assert rows == [[exp.experiment_name, "-99.0"], [exp.experiment_name, "-98.0"]]
    # info[info['termination']] indexes a counter, as main.py:110 needs
    assert info[info["termination"]] == 40


def test_reference_recorded_headers_match():
    """The headers above are the reference's own (only checked where a checkout of the reference is found, see
    oracle/ref_shim.py)."""
    from oracle import ref_shim
    base = ref_shim.fixture_dir(1)
    if not os.path.isdir(base):
        import pytest
        pytest.skip("the reference's recorded experiments are not available (set SAC_REFERENCE_ROOT)")
    from sac_agent_b200 import experiment as E
    assert open(os.path.join(base, "console.csv")).readline().strip().split(";") == E.CONSOLE_COLUMNS
    assert open(os.path.join(base, "terminations.csv")).readline().strip().split(";") == E.INFO_KEYS


def test_saved_configs_carry_every_reference_key(tmp_path):
    """A default run's tuned_configs.yaml must be readable by the reference's post-processing, which slices with
    base_settings.avg_lookback (rendering/boat_env_render.py:31, postprocessing/replayer.py:52): every key of the
    reference's configs/original_config.yaml is present with the shipped value, also for a partial config."""
    exp = S.Experiment(root=str(tmp_path), rng=random.Random(1))
    tuned = exp.save_configs()                                     # config.DEFAULTS
    assert isinstance(tuned.base_settings.avg_lookback, int) and tuned.base_settings.avg_lookback == 50
    assert tuned.base_settings.n_games == 250 and tuned.base_settings.render_skip_size == 50
    assert tuned.boat.n_max == 30 and tuned.agent.layer1_size == 256 and tuned.boat.a == 4.252
    scores = list(range(100))
    assert scores[-tuned.base_settings.avg_lookback:] == scores[50:]   # the slice replayer.py:52 takes
    exp2 = S.Experiment(experiment_name="second", root=str(tmp_path), rng=random.Random(2))
    partial = {"base_settings": {"experiment": 3, "dt": 0.25, "t_max": 2500, "test_mode": 0}, "wind": {"max_velocity": 0.4}}
    t2 = exp2.save_configs(partial)
    assert t2.base_settings.experiment == 3 and t2.base_settings.avg_lookback == 50 and t2.wind.max_velocity == 0.4
    # the defaults hold the reference's shipped values wherever tests/golden recorded them
    from boat_testlib import reference_config_record
    for sec, values in reference_config_record().items():
        for k, v in values.items():
            assert S.config.DEFAULTS[sec][k] == v, (sec, k)
