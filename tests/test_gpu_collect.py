"""The fused collection kernel (boatagent_collect, csrc/rollout.cu; TensorCorePolicy.collect, ContinuousAgent.collect,
examples/train_sac.py --collect-steps) against the loop it fuses: TensorCorePolicy.act, then
ReplayBuffer.step_store on an auto-resetting env, once per step.

Bit-equal is the expected outcome everywhere: both paths run the same forward pass, the same Philox draw and the same
fp32 sub-step, and the kernel sets up new episodes and spline pieces with the step kernel's own warp-cooperative
mapping.  The one exception is the fp64 return sums of the episode counters: they are atomics, so their rounding
depends on the order in which envs finish, in either path; the episode counts are compared exactly.

Every test but the driver's argument checks needs a B200 and is ``@pytest.mark.gpu``."""
import importlib.util
import os

import numpy as np
import pytest

from boat_testlib import ROOT

COUNTER_BYTES = 32 * 32 * 8   # the counter rows at the end of an export_state blob (kCounterSlots x 32 doubles)
COUNTS = ("reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken", "episodes")


@pytest.fixture(scope="module")
def S():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import sac_agent_b200 as pkg
    pkg.lib()
    return pkg


def make_actor(seed):
    """A seeded default init: it breaks the rudder or leaves the track within ~70 steps (experiment 6)."""
    import torch
    from sac_agent_b200.networks import ActorNetwork
    torch.manual_seed(seed)
    return ActorNetwork(None, (11,), max_action=[1.0]).cuda()


def policy(actor, seed=7):
    from sac_agent_b200.networks import TensorCorePolicy
    return TensorCorePolicy(actor, seed=seed)


def make_env(S, exp, n, seed=3, env_id_offset=0, auto_reset=True, precision="fp32"):
    cfg = S.load_config(base_settings__experiment=exp)
    env = S.BatchedBoatEnv(cfg, n, seed=seed, precision=precision, device=0, env_id_offset=env_id_offset,
                           auto_reset=auto_reset)
    env.reset()
    return env


def make_ring(S, size, obs_dim=11, n_actions=1, precision="fp32"):
    return S.ReplayBuffer(size, (obs_dim,), n_actions, precision=precision, device=0, as_torch=True)


def set_mem_cntr(mem, value):
    from sac_agent_b200 import _lib
    _lib.check(mem._L.boatreplay_set_mem_cntr(mem._h, int(value)), "boatreplay_set_mem_cntr")


def per_step(env, mem, pol, steps, done_flag_mode=1):
    for _ in range(steps):
        a = pol.act(env.obs)
        mem.step_store(env, a.reshape(-1), done_flag_mode=done_flag_mode)


def same(x, y):
    import torch
    if x.dtype == torch.float32:
        x, y = x.contiguous().view(torch.int32), y.contiguous().view(torch.int32)
    return x.shape == y.shape and torch.equal(x, y)


def ring_rows(mem):
    """Every written slot of the ring: (state, action, reward, new_state, terminal)."""
    import torch
    n = min(mem.mem_cntr, mem.mem_size)
    return mem.gather(torch.arange(n, dtype=torch.int64, device=mem.device), as_torch=True)


def state_part(env):
    return env.state_dict()["blob"][:-COUNTER_BYTES]


def assert_same_run(env_f, mem_f, pol_f, env_e, mem_e, pol_e):
    assert mem_f.mem_cntr == mem_e.mem_cntr
    for k, (x, y) in enumerate(zip(ring_rows(mem_f), ring_rows(mem_e))):
        assert same(x, y), ("state", "action", "reward", "new_state", "terminal")[k]
    for name in ("obs", "reward", "done", "term"):
        assert same(getattr(env_f, name), getattr(env_e, name)), name
    assert same(state_part(env_f), state_part(env_e))   # dyn slots, step index, wind coefficients, episode numbers
    cf, ce = env_f.counters(), env_e.counters()
    for k in COUNTS:
        assert cf[k] == ce[k], k
    for k in ("return_sum", "return_sumsq"):
        assert cf[k] == pytest.approx(ce[k], rel=1e-9, abs=1e-6), k
    assert pol_f.steps == pol_e.steps


# ---------------------------------------------------------------------------------------
# 1. bit parity with the per-step path, with several resets per env inside the call
# ---------------------------------------------------------------------------------------
CASES = [(e, 1000, 1) for e in range(1, 7)] + [(6, 1000, 0), (2, 70000, 1), (6, 70000, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("exp,n_envs,done_flag_mode", CASES)
def test_collect_matches_per_step_path(S, exp, n_envs, done_flag_mode):
    T = 400
    actor = make_actor(seed=1)
    env_f, env_e = make_env(S, exp, n_envs), make_env(S, exp, n_envs)
    mem_f, mem_e = make_ring(S, T * n_envs + 123), make_ring(S, T * n_envs + 123)
    pol_f, pol_e = policy(actor), policy(actor)
    out = pol_f.collect(env_f, mem_f, T, done_flag_mode=done_flag_mode)
    assert out[0] is env_f.obs and out[3]["term"] is env_f.term
    per_step(env_e, mem_e, pol_e, T, done_flag_mode)
    assert mem_f.mem_cntr == T * n_envs and pol_f.steps == T
    assert_same_run(env_f, mem_f, pol_f, env_e, mem_e, pol_e)
    assert env_f.counters()["episodes"] > n_envs   # resets and new episodes ran inside the call
    if done_flag_mode == 0:   # (the random actor never reaches the goal: mode 1 stores no terminal rows)
        assert bool(ring_rows(mem_f)[4].any())
    for x in (env_f, env_e, mem_f, mem_e):
        x.close()


# ---------------------------------------------------------------------------------------
# 2. chunking: the write-back (episode numbers included) lets a second call continue exactly
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_collect_chunks_continue_exactly(S):
    n = 3000
    actor = make_actor(seed=11)
    env_a, env_b = make_env(S, 6, n), make_env(S, 6, n)
    mem_a, mem_b = make_ring(S, 400 * n), make_ring(S, 400 * n)
    pol_a, pol_b = policy(actor), policy(actor)
    pol_a.collect(env_a, mem_a, 400)
    pol_b.collect(env_b, mem_b, 150)
    pol_b.collect(env_b, mem_b, 250)
    assert_same_run(env_b, mem_b, pol_b, env_a, mem_a, pol_a)
    for x in (env_a, env_b, mem_a, mem_b):
        x.close()


# ---------------------------------------------------------------------------------------
# 3. ring placement: a call that wraps the ring end; a call that would lap it is rejected and changes nothing
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_collect_wraps_the_ring(S):
    n, T = 1000, 50
    size = T * n + 333                           # not a multiple of n: rows of one step straddle the end
    actor = make_actor(seed=4)
    env_f, env_e = make_env(S, 4, n), make_env(S, 4, n)
    mem_f, mem_e = make_ring(S, size), make_ring(S, size)
    start = 3 * size - 20 * n - 517              # the call crosses the end of the ring after ~20 steps
    set_mem_cntr(mem_f, start)
    set_mem_cntr(mem_e, start)
    pol_f, pol_e = policy(actor), policy(actor)
    pol_f.collect(env_f, mem_f, T)
    per_step(env_e, mem_e, pol_e, T)
    assert mem_f.mem_cntr == start + T * n
    assert_same_run(env_f, mem_f, pol_f, env_e, mem_e, pol_e)
    for x in (env_f, env_e, mem_f, mem_e):
        x.close()


@pytest.mark.gpu
def test_collect_rejects_lapping_the_ring(S):
    import torch
    n = 1000
    pol = policy(make_actor(seed=2))
    env = make_env(S, 6, n)
    mem = make_ring(S, 10 * n + 5)
    pol.collect(env, mem, 4)
    before = ring_rows(mem), state_part(env).clone(), env.obs.clone(), mem.mem_cntr, pol.steps
    with pytest.raises(ValueError):
        pol.collect(env, mem, 11)
    rc = pol._L.boatagent_collect(env._h, mem._h, pol.blob.data_ptr(), pol.actor.max_action.data_ptr(), 7, pol.steps,
                                  11, 1, env.obs.data_ptr(), env.reward.data_ptr(), env.done.data_ptr(),
                                  env.term.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == -1                              # BOATENV_EINVAL
    torch.cuda.synchronize()
    assert mem.mem_cntr == before[3] and pol.steps == before[4]
    assert all(same(x, y) for x, y in zip(ring_rows(mem), before[0]))
    assert same(state_part(env), before[1]) and same(env.obs, before[2])
    pol.collect(env, mem, 6)                     # exactly fills the rest of the ring: accepted
    assert mem.mem_cntr == 10 * n
    env.close()
    mem.close()


# ---------------------------------------------------------------------------------------
# 4. a shard of a larger population (env_id_offset != 0) draws its own envs' episodes
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_collect_sharded_handle(S):
    n, T = 1500, 300
    actor = make_actor(seed=5)
    env_f, env_e = make_env(S, 6, n, env_id_offset=5000), make_env(S, 6, n, env_id_offset=5000)
    mem_f, mem_e = make_ring(S, T * n), make_ring(S, T * n)
    pol_f, pol_e = policy(actor), policy(actor)
    pol_f.collect(env_f, mem_f, T)
    per_step(env_e, mem_e, pol_e, T)
    assert_same_run(env_f, mem_f, pol_f, env_e, mem_e, pol_e)
    for x in (env_f, env_e, mem_f, mem_e):
        x.close()


# ---------------------------------------------------------------------------------------
# 5. with learning in between: the agent's collect is the choose_action + step_and_remember loop
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_agent_collect_with_learning_matches_per_step_loop(S):
    import torch
    from sac_agent_b200 import ContinuousAgent
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
    runs = []
    for fused in (True, False):
        torch.manual_seed(21)
        env = S.BatchedBoatEnv(cfg, 512, seed=9, precision="fp32", device=0, auto_reset=True)
        mem = make_ring(S, 30_000)
        agent = ContinuousAgent(cfg, None, (11,), env, device=0, seed=9, memory=mem, policy_precision="tcgen05")
        env.reset()
        torch.manual_seed(22)                    # the learner's Gaussian draws
        losses = []
        for _ in range(3):
            if fused:
                agent.collect(env, 4)
            else:
                for _ in range(4):
                    actions = agent.choose_action_graphed(env.obs).squeeze(-1)
                    agent.step_and_remember(env, actions)
            for _ in range(4):
                out = agent.learn()
                assert out is not None
                losses.append(torch.stack([x.clone() for x in out]))
        torch.cuda.synchronize()
        weights = [p.detach().clone() for net in agent.learner.networks() for p in net.parameters()]
        runs.append((torch.stack(losses), weights, ring_rows(mem), mem.mem_cntr, env.obs.clone()))
        env.close()
    (la, wa, ra, ca, oa), (lb, wb, rb, cb, ob) = runs
    assert ca == cb == 3 * 4 * 512
    assert same(la, lb)
    assert all(same(x, y) for x, y in zip(wa, wb))
    assert all(same(x, y) for x, y in zip(ra, rb))
    assert same(oa, ob)


# ---------------------------------------------------------------------------------------
# 6. errors
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_collect_error_codes(S):
    import torch
    pol = policy(make_actor(seed=1))
    L = pol._L
    st = torch.cuda.current_stream().cuda_stream
    env = make_env(S, 6, 64)
    mem = make_ring(S, 10_000)

    def call(e=env, m=mem, blob=None, steps=4, mode=1, obs=True, done=True, term=True):
        return L.boatagent_collect(e._h, m._h, pol.blob.data_ptr() if blob is None else blob,
                                   pol.actor.max_action.data_ptr(), 7, 0, steps, mode,
                                   e.obs.data_ptr() if obs else None, e.reward.data_ptr(),
                                   e.done.data_ptr() if done else None, e.term.data_ptr() if term else None, st)

    env64 = make_env(S, 6, 64, precision="fp64")
    assert call(e=env64) == -4                   # BOATENV_EUNSUPPORTED: fp64 handle
    for m in (make_ring(S, 10_000, precision="fp64"), make_ring(S, 10_000, obs_dim=5), make_ring(S, 10_000, n_actions=2)):
        assert call(m=m) == -4                   # ring not fp32 / obs_dim 11 / one action
        m.close()
    fresh = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), 64, precision="fp32", device=0)
    assert call(e=fresh) == -6                   # BOATENV_ESTATE: before reset
    assert call(obs=False) == -1                 # BOATENV_EINVAL
    assert call(done=False, term=False) == -1
    assert call(steps=0) == -1
    assert call(mode=2) == -1
    assert call(steps=10_000 // 64 + 1) == -1    # steps * n_envs > mem_size
    assert call(blob=pol.blob.data_ptr() + 8) == -7   # BOATENV_EALIGN
    assert mem.mem_cntr == 0
    assert call(done=False) == 0 and call(term=False) == 0   # one of the two may be NULL
    torch.cuda.synchronize()
    assert mem.mem_cntr == 2 * 4 * 64
    for x in (env, env64, fresh, mem):
        x.close()


@pytest.mark.gpu
def test_collect_value_errors(S):
    from sac_agent_b200 import ContinuousAgent
    pol = policy(make_actor(seed=1))
    mem = make_ring(S, 10_000)
    no_reset = make_env(S, 6, 64, auto_reset=False)
    with pytest.raises(ValueError):
        pol.collect(no_reset, mem, 4)
    env64 = make_env(S, 6, 64, precision="fp64")
    with pytest.raises(ValueError):
        pol.collect(env64, mem, 4)
    env = make_env(S, 6, 64)
    mem64 = make_ring(S, 10_000, precision="fp64")
    with pytest.raises(ValueError):
        pol.collect(env, mem64, 4)
    with pytest.raises(ValueError):
        pol.collect(env, mem, 10_000 // 64 + 1)
    assert mem.mem_cntr == 0 and pol.steps == 0
    cfg = S.load_config(base_settings__experiment=6)
    agent = ContinuousAgent(cfg, None, (11,), env, device=0, memory=mem, policy_precision="fp32")
    with pytest.raises(ValueError):
        agent.collect(env, 4)
    for x in (mem, no_reset, env64, env, mem64):
        x.close()


# ---------------------------------------------------------------------------------------
# 7. the driver
# ---------------------------------------------------------------------------------------
def _train_sac():
    spec = importlib.util.spec_from_file_location("train_sac", os.path.join(ROOT, "examples", "train_sac.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.gpu
def test_train_sac_collect_steps(S, monkeypatch):
    counters = []

    class Ring(S.ReplayBuffer):
        def close(self):
            if getattr(self, "_h", None):
                counters.append(self.mem_cntr)
            super().close()

    monkeypatch.setattr(S, "ReplayBuffer", Ring)
    out = _train_sac().main(["--envs", "2048", "--iters", "6", "--warmup-iters", "2", "--experiment", "6",
                             "--policy-precision", "tcgen05", "--collect-steps", "4", "--updates-per-iter", "4",
                             "--buffer", "200000", "--log-every", "0"])
    assert out["collect_steps"] == 4 and out["policy_precision"] == "tcgen05"
    assert counters == [(6 + 2) * 4 * 2048]
    assert out["env_steps_per_s"] == pytest.approx(6 * 4 * 2048 / (out["ms_per_iter"] * 6 * 1e-3))
    assert out["losses_v_pi_q"] is not None and all(np.isfinite(out["losses_v_pi_q"]))


@pytest.mark.parametrize("extra", [[], ["--policy-precision", "tcgen05", "--overlap"],
                                   ["--policy-precision", "tcgen05", "--record-envs", "2", "--experiments-root", "x"]],
                         ids=["no_tcgen05", "overlap", "record_envs"])
def test_train_sac_collect_steps_rejected_combinations(extra, capsys):
    with pytest.raises(SystemExit) as ex:
        _train_sac().main(["--envs", "64", "--iters", "1", "--collect-steps", "4"] + extra)
    assert ex.value.code == 2
    assert "--collect-steps" in capsys.readouterr().err
