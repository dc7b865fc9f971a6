"""Shared helpers of the test-suite (golden loading, the parity error metric)."""
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# observation normalisers of the reference (boat_env.py:310-321): the scale S_i of the
# error metric |a-b| / max(|b|, S_i) (SURVEY.md H6) -- applied to NORMALISED obs
# these scales are all 1; applied to raw quantities they are the spans below.
RAW_SCALES = dict(s_x=3900.0, v_x=5.0, a_x=0.025, s_y=800.0, v_y=2.0, a_y=0.37,
                  s_r=2 * np.pi, v_r=8.5e-3, a_r=1.4e-5, rudder=np.pi / 3, fuel=15000.0)


def load_golden(name):
    d = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    out = {k: d[k] for k in d.files}
    for k in ("config", "meta", "columns"):
        if k in out:
            out[k] = json.loads(str(out[k]))
    return out


AGENT_KEYS = ("learning_rate_alpha", "learning_rate_beta", "gamma", "tvn_parameter_modulation_tau", "reward_scale")


def reference_config_record():
    """The values of the reference's configs/original_config.yaml that tests/golden recorded (oracle/make_golden.py,
    make_agent_golden.py): the hot-path keys stored beside the reference roll-outs, which set
    base_settings.experiment per file (left out here), and the agent keys of the recorded SAC update."""
    cfgs = [load_golden(f"ref_rollout_exp{e}")["config"] for e in range(1, 7)]
    for e, cfg in enumerate(cfgs, 1):
        assert cfg["base_settings"].pop("experiment") == e
    assert all(cfg == cfgs[0] for cfg in cfgs)
    rec = np.load(os.path.join(GOLDEN, "agent_update.npz"))
    cfgs[0]["agent"] = {k: rec["meta/" + k].item() for k in AGENT_KEYS}
    return cfgs[0]


def scaled_err(a, b, scale=1.0):
    """|a-b| / max(|b|, scale): the parity metric of SURVEY.md H6."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), scale)
