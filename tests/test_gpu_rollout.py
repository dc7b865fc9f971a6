"""The fused policy + env rollout (boatagent_rollout, csrc/rollout.cu; TensorCorePolicy.rollout,
ContinuousAgent.evaluate, examples/evaluate_sac.py) against the per-step path it fuses: TensorCorePolicy.act then
BatchedBoatEnv.step without auto-reset.  Needs a B200: every test is ``@pytest.mark.gpu``.

Bit-equal is the expected outcome everywhere: both paths run the same forward pass, the same Philox draw and the
same fp32 sub-step, and the piece-change setup of the rollout (one env per lane) computes the same coefficients as
the step kernel's (warp-cooperative / setup warps, wind_setup.cuh)."""
import json
import os
import sys

import numpy as np
import pytest

from boat_testlib import ROOT, load_golden

pytestmark = pytest.mark.gpu

FIELDS = ("v_x", "v_y", "v_r", "rudder_angle", "s_x", "s_y", "s_r", "episode_reward", "index", "episode")


@pytest.fixture(scope="module")
def S():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import sac_agent_b200 as pkg
    pkg.lib()
    return pkg


def make_actor(kind, seed=0):
    """'random': seeded default init; 'zero': mean head zero (action exactly 0 when deterministic);
    'low_noise': mean head zero, std-head bias -20 (log_std -> -5: small steering noise, long episodes)."""
    import torch
    from sac_agent_b200.networks import ActorNetwork
    torch.manual_seed(seed)
    actor = ActorNetwork(None, (11,), max_action=[1.0]).cuda()
    with torch.no_grad():
        if kind in ("zero", "low_noise"):
            actor.mean.weight.zero_()
            actor.mean.bias.zero_()
        if kind == "low_noise":
            actor.std.bias.fill_(-20.0)
    return actor


def policy(actor, seed=7):
    from sac_agent_b200.networks import TensorCorePolicy
    return TensorCorePolicy(actor, seed=seed)


def make_env(S, exp, n, seed=3, env_id_offset=0):
    cfg = S.load_config(base_settings__experiment=exp)
    env = S.BatchedBoatEnv(cfg, n, seed=seed, precision="fp32", device=0, env_id_offset=env_id_offset, auto_reset=False)
    env.reset()
    return env


def counts(env):
    c = env.counters()
    return np.array([c[k] for k in ("reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken",
                                    "episodes")])


def hist(term):
    t = term.cpu().numpy()
    return np.array([np.sum(t == k) for k in range(1, 6)] + [np.sum(t != 0)], dtype=np.float64)


def eager(env, pol, max_steps, deterministic):
    """The per-step loop up to each env's first termination: (returns, steps, term, obs) as the rollout reports them."""
    import torch
    n, dev = env.n_envs, env.device
    ret = torch.zeros(n, dtype=torch.float32, device=dev)
    steps = torch.zeros(n, dtype=torch.int32, device=dev)
    term = torch.zeros(n, dtype=torch.uint8, device=dev)
    fin = torch.zeros((n, 11), dtype=torch.float32, device=dev)
    ended = torch.zeros(n, dtype=torch.bool, device=dev)
    eps = torch.zeros((n, 1), dtype=torch.float32, device=dev) if deterministic else None
    for t in range(max_steps):
        a = pol.act(env.obs, eps=eps)
        obs, rew, _, info = env.step(a.reshape(-1))
        live = ~ended
        ret = torch.where(live, ret + rew, ret)
        steps += live.to(torch.int32)
        newly = live & (info["term"] != 0)
        term = torch.where(newly, info["term"], term)
        fin = torch.where(newly[:, None], obs, fin)
        ended |= newly
        if t % 64 == 63 and bool(ended.all()):
            pol.steps += max_steps - 1 - t
            break
    fin = torch.where(ended[:, None], fin, env.obs)
    return ret, steps, term, fin


def bits(t):
    import torch
    return t.contiguous().view(torch.int32).cpu().numpy() if t.dtype == torch.float32 else t.cpu().numpy()


# ---------------------------------------------------------------------------------------
# 1. known answer: the reference's recorded fixtures, action exactly 0
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_envs", [1, 300])
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6])
def test_rollout_recorded_fixture(S, n, n_envs):
    g = load_golden(f"fixture_exp{n}")
    fp = int(g["config"]["wind"]["fixed_points"])
    knots = np.zeros((1, 2, fp))
    if g["meta"]["kind_v"] == "curve":
        knots[0, 0] = g["knots_v"]
    if g["meta"]["kind_a"] == "curve":
        knots[0, 1] = g["knots_a"]
    if g["meta"]["kind_a"] == "rect":
        knots[0, 0] = g["knots_r"]
    env = S.BatchedBoatEnv(g["config"], n_envs, precision="fp32", device=0, auto_reset=False)
    env.set_episode_draws(np.full(n_envs, int(g["s_y_start"])), np.repeat(knots, n_envs, axis=0))
    env.reset()
    before = counts(env)
    ret, steps, term = policy(make_actor("zero")).rollout(env, 6000, deterministic=True)
    assert (steps.cpu().numpy() == int(g["n_rows"])).all()
    assert (term.cpu().numpy() == 1).all() and str(g["termination"]) == "reached_goal"
    if n == 6:
        assert np.abs(ret.double().cpu().numpy() - 871.2727580297085).max() <= 0.05
    assert np.array_equal(counts(env) - before, hist(term))
    env.close()


# ---------------------------------------------------------------------------------------
# 2. bit parity with the per-step path
# ---------------------------------------------------------------------------------------
ACTORS = [("random", False, 1000), ("random", True, 1000), ("low_noise", False, 5000)]


@pytest.mark.parametrize("n_envs", [1000, 70000])
@pytest.mark.parametrize("exp", [1, 2, 6])
@pytest.mark.parametrize("actor_kind,deterministic,max_steps", ACTORS)
def test_rollout_matches_per_step_path(S, exp, n_envs, actor_kind, deterministic, max_steps):
    actor = make_actor(actor_kind, seed=exp)
    env_f, env_e = make_env(S, exp, n_envs), make_env(S, exp, n_envs)
    before = counts(env_f)
    pol_f, pol_e = policy(actor), policy(actor)
    ret, steps, term = pol_f.rollout(env_f, max_steps, deterministic=deterministic)
    e_ret, e_steps, e_term, e_obs = eager(env_e, pol_e, max_steps, deterministic)
    assert pol_f.steps == pol_e.steps == max_steps
    assert np.array_equal(bits(term), bits(e_term))
    assert np.array_equal(bits(steps), bits(e_steps))
    assert np.array_equal(bits(ret), bits(e_ret))
    assert np.array_equal(bits(env_f.obs), bits(e_obs))
    running = term.cpu().numpy() == 0
    for f in FIELDS:
        assert np.array_equal(bits(env_f.get_field(f))[running], bits(env_e.get_field(f))[running]), f
    assert np.array_equal(counts(env_f) - before, hist(term))
    if actor_kind == "low_noise":   # long episodes: thousands of steps, several spline-piece changes (exp 6)
        assert steps.float().mean().item() > 3000
    env_f.close()
    env_e.close()


# ---------------------------------------------------------------------------------------
# 3. chunking: the write-back lets a second rollout continue exactly
# ---------------------------------------------------------------------------------------
def test_rollout_chunks_continue_exactly(S):
    actor = make_actor("low_noise", seed=11)
    env_a, env_b = make_env(S, 6, 4096), make_env(S, 6, 4096)
    ret, steps, term = policy(actor).rollout(env_a, 2000)
    pol_b = policy(actor)
    _, steps1, term1 = pol_b.rollout(env_b, 1000)
    ret2, steps2, term2 = pol_b.rollout(env_b, 1000)
    assert (term1.cpu().numpy() == 0).all()   # nobody ends in the first chunk: the two runs step the same envs
    assert np.array_equal(bits(term2), bits(term))
    assert np.array_equal(bits(steps1 + steps2), bits(steps))
    assert np.array_equal(bits(ret2), bits(ret))
    assert np.array_equal(bits(env_b.obs), bits(env_a.obs))
    for f in FIELDS:
        assert np.array_equal(bits(env_b.get_field(f)), bits(env_a.get_field(f))), f
    ca, cb = env_a.counters(), env_b.counters()
    for k in ("reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken", "episodes"):
        assert ca[k] == cb[k]
    # and the per-step path continues from the rollout's state like from its own
    import torch
    a = torch.zeros(4096, dtype=torch.float32, device=env_a.device)
    oa = env_a.step(a)[0].clone()
    ob = env_b.step(a)[0].clone()
    assert np.array_equal(bits(oa), bits(ob))
    env_a.close()
    env_b.close()


# ---------------------------------------------------------------------------------------
# 4. sharding: deterministic mode is independent of how the envs are split over handles
# ---------------------------------------------------------------------------------------
def test_rollout_shards_match_one_handle(S):
    import torch
    n = 3000
    actor = make_actor("random", seed=5)
    full = make_env(S, 6, n)
    halves = [make_env(S, 6, n // 2, env_id_offset=0), make_env(S, 6, n - n // 2, env_id_offset=n // 2)]
    ret, steps, term = policy(actor).rollout(full, 1500, deterministic=True)
    parts = [policy(actor).rollout(h, 1500, deterministic=True) for h in halves]
    assert np.array_equal(bits(ret), bits(torch.cat([p[0] for p in parts])))
    assert np.array_equal(bits(steps), bits(torch.cat([p[1] for p in parts])))
    assert np.array_equal(bits(term), bits(torch.cat([p[2] for p in parts])))
    assert np.array_equal(bits(full.obs), bits(torch.cat([h.obs for h in halves])))
    for e in [full] + halves:
        e.close()


# ---------------------------------------------------------------------------------------
# 5. errors
# ---------------------------------------------------------------------------------------
def test_rollout_errors(S):
    import torch
    from sac_agent_b200 import _lib
    pol = policy(make_actor("random"))
    cfg = S.load_config(base_settings__experiment=6)
    env64 = S.BatchedBoatEnv(cfg, 64, precision="fp64", device=0, auto_reset=False)
    env64.reset()
    with pytest.raises(S.BoatEnvError) as ex:
        pol.rollout(env64, 10)
    assert ex.value.code == -4   # BOATENV_EUNSUPPORTED
    env = S.BatchedBoatEnv(cfg, 64, precision="fp32", device=0, auto_reset=False)
    with pytest.raises(S.BoatEnvError) as ex:
        pol.rollout(env, 10)
    assert ex.value.code == -6   # BOATENV_ESTATE
    env.reset()
    with pytest.raises(S.BoatEnvError) as ex:
        pol.rollout(env, 0)
    assert ex.value.code == -1   # BOATENV_EINVAL
    L = _lib.lib()
    dev = torch.cuda.current_stream().cuda_stream
    out = torch.empty(64, dtype=torch.float32, device=env.device)
    rc = L.boatagent_rollout(env._h, pol.blob.data_ptr(), pol.actor.max_action.data_ptr(), 0, 0, 10, 0,
                             env.obs.data_ptr(), env.obs.data_ptr(), out.data_ptr(), None, None, dev)
    with pytest.raises(S.BoatEnvError) as ex:
        _lib.check(rc, "boatagent_rollout")
    assert ex.value.code == -1
    rc = L.boatagent_rollout(env._h, pol.blob.data_ptr() + 8, pol.actor.max_action.data_ptr(), 0, 0, 10, 0,
                             env.obs.data_ptr(), env.obs.data_ptr(), out.data_ptr(), out.data_ptr(), out.data_ptr(), dev)
    assert rc == -7             # BOATENV_EALIGN
    env.close()
    env64.close()


# ---------------------------------------------------------------------------------------
# 6. the agent and the example
# ---------------------------------------------------------------------------------------
def _examples():
    p = os.path.join(ROOT, "examples")
    if p not in sys.path:
        sys.path.insert(0, p)
    import evaluate_sac
    import train_sac
    return train_sac, evaluate_sac


def test_evaluate_sac_example(S, tmp_path, capsys):
    train_sac, evaluate_sac = _examples()
    root = str(tmp_path / "exp")
    train_sac.main(["--envs", "2048", "--iters", "400", "--warmup-iters", "0", "--experiment", "6",
                    "--experiments-root", root, "--log-every", "100", "--buffer", "200000"])
    capsys.readouterr()
    dirs = [dp for dp, dn, fn in os.walk(root) if "checkpoints" in dn]
    assert len(dirs) == 1
    ckpt = dirs[0]
    evaluate_sac.main(["--checkpoints", ckpt, "--envs", "500", "--experiment", "6", "--rounds", "2",
                       "--max-steps", "3000"])
    summary = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert summary["envs"] == 500 and summary["rounds"] == 2
    assert summary["episodes"] + summary["running"] == 1000
    assert sum(summary["terminations"].values()) == summary["episodes"]

    rec = tmp_path / "rec"
    evaluate_sac.main(["--checkpoints", ckpt, "--envs", "64", "--experiment", "6", "--max-steps", "6000",
                       "--record-envs", "2", "--output", str(rec), "--stochastic"])
    summary = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert summary["recorded_envs"] == 2
    for i, (steps, term) in enumerate(zip(summary["recorded_steps"], summary["recorded_term"])):
        data = (rec / "episodes" / f"env{i}_episode_0_data.csv").read_text().strip().splitlines()
        # header, the reset state, then one row per step; the terminal state is never written (main.py:79-81)
        assert len(data) - 1 == (steps if term else steps + 1)
        assert not (rec / "episodes" / f"env{i}_episode_1_data.csv").exists()
        if term:
            info = (rec / "episodes" / f"env{i}_info.csv").read_text().strip().splitlines()
            assert len(info) == 2 and S.TERM_NAMES[term] in info[1]
