"""The episode statistics against the CPU oracle: the eight counters of every env handle (the five termination kinds,
``episodes``, ``return_sum``, ``return_sumsq``), the per-env running return (the ``episode_reward`` field), the rollout
kernel's ``return_out``, and what ``sharding.all_reduce_counters`` and ``experiment.info_from_counters`` make of them.

Every expected value is built from the oracle's per-step output by ``episode_reference``: each env's steps are split
into episodes at ``done``, and an episode's return is the float64 sum of its rewards in step order, which is the
reference's ``info['episode_reward']`` (boat_env.py:113).  No case passes because two kernels agree.

Tolerances (derived, not fitted):
  * termination counts and ``episodes``: exact.
  * one episode, fp32 mode: the fp32 running sum rounds once per step (<= |partial sum| 2^-24) and each step's
    reward carries the fp32 parity tolerance TOL32 max(1, |r|) of test_gpu_parity.py, so
    |err| <= sum_t (|partial_t| 2^-24 + TOL32 max(1, |r_t|)).
  * one episode, fp64 mode: the fp64 step follows the reference's operation order; the per-step term is
    STEP64 max(1, |r_t|) with STEP64 = 1e-13 (observations match the oracle to <= 2.5e-14, DESIGN.md section 4) and
    the rounding term |partial_t| 2^-52.
  * ``return_sum`` / ``return_sumsq``: the counter rows are summed with fp64 atomics in no fixed order, which adds
    (n + 32) 2^-52 sum|x| (resp. sum x^2) on top of the per-episode bounds (n episodes, 32 counter rows).
The tests print the worst measured error as a fraction of its bound.

Tests without the ``gpu`` mark run the reference and the choice of actions on the CPU.
"""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from boat_testlib import ROOT, load_golden

TOL32 = 1e-4      # fp32 per-step reward tolerance (test_gpu_parity.py)
STEP64 = 1e-13    # fp64 per-step reward tolerance of the return bounds (see the module docstring)
U32, U64 = 2.0 ** -24, 2.0 ** -52
KINDS = ("reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken")
COUNTER_ROWS = 32


@pytest.fixture(scope="module")
def S():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import sac_agent_b200 as pkg
    pkg.lib()
    return pkg


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def pkg():
    import sac_agent_b200
    return sac_agent_b200


def np_(t):
    return t.detach().double().cpu().numpy() if t.is_floating_point() else t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
# the host reference
# ---------------------------------------------------------------------------------------------------------------------
def episode_reference(reward, done, term, auto_reset=True, valid=None, restart=None):
    """Episode statistics of the oracle's per-step output (reward / done / term [T, N]).

    auto_reset: a done step starts a new episode (return 0).  Without it the reference object keeps its cumulative
      ``info``: every done step counts its kind again, with ``episode_reward`` = the sum since the last reset().
    valid [T, N]: the steps that were executed (K-step windows stop an env at its first done); default all.
    restart [T, N]: a reset() before that step that ends no episode (masked reset of a live env).

    Returns a dict: counts [8] (the counter vector), returns / kinds / bound32 / bound64 of the finished episodes (in
    the order they finish), running [T, N] = the per-env running return after each step (the ``episode_reward``
    field), and its bounds run32 / run64 [T, N]."""
    reward = np.asarray(reward, dtype=np.float64)
    done = np.asarray(done).astype(bool)
    T, N = reward.shape
    run, b32, b64 = np.zeros(N), np.zeros(N), np.zeros(N)
    rets, kinds, e32, e64 = [], [], [], []
    running, run32, run64 = np.empty((T, N)), np.empty((T, N)), np.empty((T, N))
    for t in range(T):
        if restart is not None and restart[t].any():
            m = np.asarray(restart[t], dtype=bool)
            run[m] = 0.0; b32[m] = 0.0; b64[m] = 0.0
        v = np.ones(N, dtype=bool) if valid is None else np.asarray(valid[t], dtype=bool)
        r = np.where(v, reward[t], 0.0)
        run = run + r                       # float64, step order: boat_env.py:113
        a, w = np.abs(run), np.maximum(1.0, np.abs(r))
        b32 = b32 + np.where(v, a * U32 + TOL32 * w, 0.0)
        b64 = b64 + np.where(v, a * U64 + STEP64 * w, 0.0)
        d = done[t] & v
        if d.any():
            rets.append(run[d].copy()); kinds.append(np.asarray(term[t])[d].astype(int))
            e32.append(b32[d].copy()); e64.append(b64[d].copy())
            if auto_reset:
                run[d] = 0.0; b32[d] = 0.0; b64[d] = 0.0
        running[t], run32[t], run64[t] = run, b32, b64
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)  # noqa: E731
    x, k = cat(rets, np.float64), cat(kinds, int)
    counts = np.array([float((k == c).sum()) for c in range(1, 6)] + [float(len(x)), math.fsum(x),
                                                                     math.fsum(x * x)])
    return dict(counts=counts, returns=x, kinds=k, bound32=cat(e32, np.float64), bound64=cat(e64, np.float64),
                running=running, run32=run32, run64=run64)


def merge(*refs):
    """The statistics of several disjoint env sets (shards) as one."""
    x = np.concatenate([r["returns"] for r in refs])
    out = dict(returns=x, kinds=np.concatenate([r["kinds"] for r in refs]),
               bound32=np.concatenate([r["bound32"] for r in refs]), bound64=np.concatenate([r["bound64"] for r in refs]))
    out["counts"] = np.array([float((out["kinds"] == c).sum()) for c in range(1, 6)] + [float(len(x)), math.fsum(x),
                                                                                       math.fsum(x * x)])
    return out


def sum_tolerances(ref, precision):
    """(tol return_sum, tol return_sumsq) of the reference's episodes."""
    x = ref["returns"]
    b = ref["bound32"] if precision == "fp32" else ref["bound64"]
    n = len(x) + COUNTER_ROWS
    tol_sum = b.sum() + n * U64 * np.abs(x).sum()
    tol_sq = (2.0 * np.abs(x) * b + b * b).sum() + n * U64 * (x * x).sum()
    return tol_sum, tol_sq


def check_counters(c, ref, precision, base=None):
    """Counter dict `c` (minus `base`, a dict of the counters before) against the reference's 8-vector."""
    got = np.array([c[k] for k in KINDS + ("episodes", "return_sum", "return_sumsq")], dtype=np.float64)
    if base is not None:
        got -= np.array([base[k] for k in KINDS + ("episodes", "return_sum", "return_sumsq")], dtype=np.float64)
    want = ref["counts"]
    assert np.array_equal(got[:6], want[:6]), (got[:6], want[:6])
    tol_sum, tol_sq = sum_tolerances(ref, precision)
    assert abs(got[6] - want[6]) <= tol_sum, (got[6], want[6], tol_sum)
    assert abs(got[7] - want[7]) <= tol_sq, (got[7], want[7], tol_sq)
    if want[5]:
        print(f"[episode statistics] counters ({precision}, {int(want[5])} episodes): |error| / bound = "
              f"{abs(got[6] - want[6]) / tol_sum:.3g} (return_sum), {abs(got[7] - want[7]) / tol_sq:.3g} (return_sumsq)")


def check_within(name, got, want, bound):
    """|got - want| <= bound elementwise; prints the worst ratio (the headroom)."""
    got, want, bound = (np.asarray(x, dtype=np.float64) for x in (got, want, bound))
    err = np.abs(got - want)
    ratio = float((err / np.where(bound > 0, bound, np.inf)).max()) if err.size else 0.0
    print(f"[episode statistics] {name}: worst |error| / bound = {ratio:.3g} over {err.size} values")
    bad = err > bound
    assert not bad.any(), (name, got[bad][:5], want[bad][:5], bound[bad][:5])
    return ratio


# ---------------------------------------------------------------------------------------------------------------------
# inputs (built on the host: the CPU tests check what they cover)
# ---------------------------------------------------------------------------------------------------------------------
def host_draws(cfg, n, episodes, seed, env_id_offset=0):
    """The Philox draws of envs [offset, offset + n), episodes 0 .. episodes-1 (boatenv_episode_draws_batch_host)."""
    import ctypes as C
    S = pkg()
    from sac_agent_b200 import _lib
    p = S.params_from_config(cfg)
    fp = int(p.fixed_points)
    ids = np.ascontiguousarray(np.arange(n, dtype=np.int64) + env_id_offset)
    s_y = np.empty((episodes, n), dtype=np.int32)
    knots = np.empty((episodes, n, 2, fp), dtype=np.float64)
    _lib.check(_lib.lib().boatenv_episode_draws_batch_host(C.byref(p), seed, ids.ctypes.data, n, 0, episodes,
                                                         s_y.ctypes.data, knots.ctypes.data), "episode_draws")
    return s_y, knots


def uniform(rng, T, n, scale):
    return (scale * rng.uniform(-1, 1, size=(T, n))).astype(np.float32)


def mixed_case(experiment):
    """Step-kernel inputs of one experiment: 1024 envs x 1200 steps with auto-reset (32 state blocks: every counter
    row).  Envs 0-511: uniform A1 actions (rudder_broken); 512-767: tiny actions (out_of_fuel at step 1000 in odd
    experiments, timeout at step 1000 in even ones); 768-1023: a hard turn to either side for 45 steps, then straight
    (out_of_bounds from experiment 2's random starts)."""
    S = pkg()
    over = dict(base_settings__experiment=experiment)
    if experiment % 2:
        over["boat__fuel"] = 999
    else:
        over["base_settings__t_max"] = 250
    cfg = S.load_config(**over)
    n, T = 1024, 1200
    rng = np.random.default_rng(100 + experiment)
    a = np.zeros((T, n), dtype=np.float32)
    a[:, :512] = uniform(rng, T, 512, 1.0)
    a[:, 512:768] = uniform(rng, T, 256, 0.01)
    a[:45, 768:] = (0.2 * np.where(np.arange(256) % 2 == 0, 1.0, -1.0)).astype(np.float32)
    s_y, knots = host_draws(cfg, n, 12, seed=experiment)
    return cfg, a, s_y, knots, experiment


def fixture_case(experiment):
    """The reference's recorded fixture of this experiment, zero actions: reached_goal after ~4960 steps, then the
    next episode (the same prescribed draws) runs on.  32 envs x 5000 steps with auto-reset."""
    g = load_golden(f"fixture_exp{experiment}")
    fp = int(g["config"]["wind"]["fixed_points"])
    knots = np.zeros((2, fp))
    if g["meta"]["kind_v"] == "curve":
        knots[0] = g["knots_v"]
    if g["meta"]["kind_a"] == "curve":
        knots[1] = g["knots_a"]
    if g["meta"]["kind_a"] == "rect":
        knots[0] = g["knots_r"]
    n, T, E = 32, 5000, 2
    s_y = np.full((E, n), int(g["s_y_start"]), dtype=np.int32)
    return g["config"], np.zeros((T, n), dtype=np.float32), s_y, np.broadcast_to(knots, (E, n, 2, fp)).copy()


def oracle_ref(O, cfg, actions, s_y, knots, auto_reset=True, n_threads=0):
    return O.rollout(O.params_from_config(cfg), np.asarray(actions, dtype=np.float64), s_y, knots,
                     auto_reset=auto_reset, n_threads=n_threads)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself, and that the chosen inputs cover every termination kind
# ---------------------------------------------------------------------------------------------------------------------
def test_episode_reference_by_hand():
    """Two envs, five steps: env 0 ends on step 1 (goal) and step 4 (rudder); env 1 never ends."""
    r = np.array([[1.0, 0.5], [1000.25, 0.5], [-2.0, 0.5], [-3.0, 0.5], [-4.0, 0.5]])
    done = np.zeros((5, 2), np.uint8); term = np.zeros((5, 2), np.uint8)
    done[1, 0], term[1, 0], done[4, 0], term[4, 0] = 1, 1, 1, 5
    ref = episode_reference(r, done, term)
    assert list(ref["returns"]) == [1001.25, -9.0] and list(ref["kinds"]) == [1, 5]
    assert list(ref["counts"]) == [1, 0, 0, 0, 1, 2, 992.25, 1001.25 ** 2 + 81.0]
    assert list(ref["running"][:, 0]) == [1.0, 0.0, -2.0, -5.0, 0.0]
    assert list(ref["running"][:, 1]) == [0.5, 1.0, 1.5, 2.0, 2.5]
    # fp32 bound of the first episode: |1| 2^-24 + 1e-4 + |1001.25| 2^-24 + 1000.25e-4
    assert ref["bound32"][0] == pytest.approx((1.0 + 1001.25) * U32 + TOL32 * (1.0 + 1000.25), rel=1e-15)
    # without auto-reset the info stays cumulative: the second done counts the whole sum since reset()
    cum = episode_reference(r, done, term, auto_reset=False)
    assert list(cum["returns"]) == [1001.25, 992.25] and list(cum["running"][:, 0]) == [1, 1001.25, 999.25, 996.25,
                                                                                         992.25]
    # a K-window stops env 0 after its done (step 2 not executed); a masked reset before step 3 drops env 1's run
    valid = np.ones((5, 2), bool); valid[2, 0] = False
    restart = np.zeros((5, 2), bool); restart[3, 1] = True
    w = episode_reference(r, done, term, valid=valid, restart=restart)
    assert list(w["returns"]) == [1001.25, -7.0] and list(w["running"][:, 1]) == [0.5, 1.0, 1.5, 0.5, 1.0]
    assert list(merge(ref, w)["counts"][:6]) == [2, 0, 0, 0, 2, 4]


def test_chosen_actions_cover_every_termination_kind(O):
    """The step-kernel cases of this file end episodes of all five kinds in the oracle."""
    total = np.zeros(5)
    for e in range(1, 7):
        cfg, a, s_y, knots, _ = mixed_case(e)
        total += episode_reference(*(oracle_ref(O, cfg, a, s_y, knots)[k] for k in ("reward", "done", "term")))[
            "counts"][:5]
    cfg, a, s_y, knots = fixture_case(6)
    ref = oracle_ref(O, cfg, a, s_y, knots)
    total += episode_reference(ref["reward"], ref["done"], ref["term"])["counts"][:5]
    assert np.all(total > 0), dict(zip(KINDS, total))


# ---------------------------------------------------------------------------------------------------------------------
# GPU drivers
# ---------------------------------------------------------------------------------------------------------------------
def make_env(S, cfg, n, precision, seed, auto_reset=True, env_id_offset=0, draws=None):
    env = S.BatchedBoatEnv(cfg, n, seed=seed, precision=precision, device=0, auto_reset=auto_reset,
                           env_id_offset=env_id_offset)
    if draws is not None:   # prescribed draws of every episode (the fixtures)
        env.set_episode_draws(draws[0][0], draws[1][0])
    env.reset()
    return env


def drive(env, actions, path="step", mem=None, done_flag_mode=1):
    """T steps of `actions` [T, N] through one of the K = 1 paths.  Returns done [T, N] and the episode_reward field
    after each step [T, N]."""
    import torch
    T, n = actions.shape
    a_dev = torch.from_numpy(np.ascontiguousarray(actions)).to(env.device).to(env.dtype)
    dones = torch.empty((T, n), dtype=torch.uint8, device=env.device)
    field = torch.empty((T, n), dtype=env.dtype, device=env.device)
    if path == "host":
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()  # noqa: E731
        act_h, obs_h, rew_h = pin(n, env.dtype), pin((n, 11), env.dtype), pin(n, env.dtype)
        done_h, term_h = pin(n, torch.uint8), pin(n, torch.uint8)
    for t in range(T):
        if path == "step":
            d = env.step(a_dev[t])[2]
        elif path == "store":
            d = mem.step_store(env, a_dev[t], done_flag_mode=done_flag_mode)[2]
        else:
            act_h.copy_(a_dev[t])
            env.step_host(act_h, obs_h, rew_h, done_h, term_h)
            d = done_h
        dones[t] = d
        field[t] = env.get_field("episode_reward")
    return np_(dones), np_(field)


def check_run(S, env, ref_out, done, field, precision, name, auto_reset=True, base=None):
    """Counters and the running return of a K = 1 run against the reference."""
    assert np.array_equal(done, ref_out["done"])
    ref = episode_reference(ref_out["reward"], ref_out["done"], ref_out["term"], auto_reset=auto_reset)
    check_counters(env.counters(), ref, precision, base)
    check_within(f"{name} running return", field, ref["running"], ref["run32" if precision == "fp32" else "run64"])
    return ref


# ---------------------------------------------------------------------------------------------------------------------
# 1. the step kernel, K = 1, auto-reset; 5. step_host
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("experiment", range(1, 7))
def test_step_counters_match_oracle(S, O, experiment, precision):
    cfg, a, s_y, knots, seed = mixed_case(experiment)
    ref_out = oracle_ref(O, cfg, a, s_y, knots)
    env = make_env(S, cfg, a.shape[1], precision, seed)
    done, field = drive(env, a)
    ref = check_run(S, env, ref_out, done, field, precision, f"step exp{experiment} {precision}")
    assert ref["counts"][5] > 1024
    env.close()
    cfg, a, s_y, knots = fixture_case(experiment)
    ref_out = oracle_ref(O, cfg, a, s_y, knots)
    env = make_env(S, cfg, a.shape[1], precision, 0, draws=(s_y, knots))
    done, field = drive(env, a)
    ref = check_run(S, env, ref_out, done, field, precision, f"fixture exp{experiment} {precision}")
    assert ref["counts"][0] == 32 and ref["counts"][5] == 32   # one goal per env, the +1000 inside its return
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("experiment", [2, 6])
def test_step_host_counters_match_oracle(S, O, experiment, precision):
    cfg, a, s_y, knots, seed = mixed_case(experiment)
    ref_out = oracle_ref(O, cfg, a, s_y, knots)
    env = make_env(S, cfg, a.shape[1], precision, seed)
    done, field = drive(env, a, path="host")
    check_run(S, env, ref_out, done, field, precision, f"step_host exp{experiment} {precision}")
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. without auto-reset, stepping past done
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_stepping_past_done_counts_like_the_cumulative_info(S, O, precision):
    """The reference object stepped on after done (boat_env.py:84-113) adds 1 to info[kind] on every done step and
    keeps adding to info['episode_reward'] until reset().  The counters do the same: every done step is one more
    episode of its kind, with the return accumulated since the last reset."""
    cfg = S.load_config(base_settings__experiment=4, boat__fuel=40)
    n, T = 64, 120
    a = uniform(np.random.default_rng(2), T, n, 0.05)
    s_y, knots = host_draws(cfg, n, 1, seed=5)
    ref_out = oracle_ref(O, cfg, a, s_y, knots, auto_reset=False)
    env = make_env(S, cfg, n, precision, 5, auto_reset=False)
    done, field = drive(env, a)
    ref = check_run(S, env, ref_out, done, field, precision, f"past done {precision}", auto_reset=False)
    assert ref["counts"][2] == n * (T - 40)   # out_of_fuel on every step after the 40th
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the fused step + ring store
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("done_flag_mode", [0, 1])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_step_store_counters_match_oracle(S, O, precision, done_flag_mode):
    cfg, a, s_y, knots, seed = mixed_case(6)
    ref_out = oracle_ref(O, cfg, a, s_y, knots)
    env = make_env(S, cfg, a.shape[1], precision, seed)
    mem = S.ReplayBuffer(3 * a.shape[1] + 5, (11,), 1, precision=precision, device=0, as_torch=True)
    done, field = drive(env, a, path="store", mem=mem, done_flag_mode=done_flag_mode)
    check_run(S, env, ref_out, done, field, precision, f"step_store mode {done_flag_mode} {precision}")
    env.close(); mem.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. step_k, K = 8; 5. step_k_host
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path,per_substep", [("device", False), ("device", True), ("host", True)])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_step_k_counters_match_oracle(S, O, precision, path, per_substep):
    """K = 8 fused sub-steps with auto-reset, emulated env by env on the oracle: an env stops at its first done in a
    window, its episode's return is the sum over all its sub-steps, the next window starts its next episode."""
    import torch
    cfg = S.load_config(base_settings__experiment=6)
    n, K, W, E = 160, 8, 60, 40
    env = make_env(S, cfg, n, precision, 31)
    s_y, knots = host_draws(cfg, n, E, seed=31)
    p = O.params_from_config(cfg)
    oracles = [O.OracleEnv(p) for _ in range(n)]
    episode = [0] * n
    for i, o in enumerate(oracles):
        o.reset(int(s_y[0, i]), knots[0, i, 0], knots[0, i, 1])
    rng = np.random.default_rng(8 if per_substep else 9)
    rew = np.zeros((W * K, n)); dn = np.zeros((W * K, n), np.uint8); tm = np.zeros((W * K, n), np.uint8)
    valid = np.zeros((W * K, n), bool)
    field = np.empty((W, n))
    ends_at = set()
    if path == "host":
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()  # noqa: E731
        act_h, obs_h, rew_h = pin((K, n), env.dtype), pin((n, 11), env.dtype), pin(n, env.dtype)
        done_h, term_h, steps_h = pin(n, torch.uint8), pin(n, torch.uint8), pin(n, torch.int32)
    for w in range(W):
        a_np = uniform(rng, K, n, 1.5) if per_substep else uniform(rng, 1, n, 1.5)[0]
        if path == "host":
            act_h.copy_(torch.from_numpy(a_np).to(env.dtype))
            env.step_k_host(act_h, K, obs_h, rew_h, done_h, term_h, steps_h)
            steps = steps_h.numpy().copy()
        else:
            steps = np_(env.step_k(torch.from_numpy(a_np).to(env.device), K)[3]["steps"])
        field[w] = np_(env.get_field("episode_reward"))
        for i, o in enumerate(oracles):
            for k in range(K):
                _, r, d, code = o.step(float(a_np[k, i] if per_substep else a_np[i]))
                row = w * K + k
                rew[row, i], dn[row, i], tm[row, i], valid[row, i] = r, d, code, True
                if d:
                    ends_at.add(k)
                    episode[i] += 1
                    o.reset(int(s_y[episode[i], i]), knots[episode[i], i, 0], knots[episode[i], i, 1])
                    break
            assert steps[i] == k + 1
    ref = episode_reference(rew, dn, tm, valid=valid)
    assert {0, K - 1} <= ends_at and ref["counts"][5] > n   # episodes end on the first and the last sub-step
    check_counters(env.counters(), ref, precision)
    last = np.arange(K - 1, W * K, K)
    check_within(f"step_k {path} per_substep={per_substep} {precision} running return", field, ref["running"][last],
                 ref["run32" if precision == "fp32" else "run64"][last])
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. the rollout kernel
# ---------------------------------------------------------------------------------------------------------------------
def constant_policy(c):
    """An actor whose deterministic action is tanh(atanh(c)) for every env and step (zero mean-head weights)."""
    import torch
    from sac_agent_b200.networks import ActorNetwork, TensorCorePolicy
    torch.manual_seed(0)
    actor = ActorNetwork(None, (11,), max_action=[1.0]).cuda()
    with torch.no_grad():
        actor.mean.weight.zero_()
        actor.mean.bias.fill_(float(np.arctanh(c)))
    return TensorCorePolicy(actor, seed=3)


ROLLOUTS = [  # name, experiment, config overrides, constant action, the kinds that must occur
    ("goal", 1, dict(boat_env__goal_line=1500), 0.0, {1}),
    ("oob", 2, {}, 2e-3, {2, 5}),
    ("timeout", 6, dict(base_settings__t_max=800), 0.0, {4}),
    ("mixed", 5, dict(base_settings__t_max=800), 1e-3, {2, 4}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,experiment,over,c,kinds", ROLLOUTS, ids=[r[0] for r in ROLLOUTS])
def test_rollout_returns_match_oracle(S, O, name, experiment, over, c, kinds):
    """return_out, steps_out, term_out and the counter deltas of a deterministic rollout with one constant action,
    then a second call on the frozen envs: the reference object stepped on after done counts the kind again, with the
    return accumulated since reset() (boat_env.py:84-113).  (A timed-out env would step past the end of the wind
    table, an IndexError in the reference: the second call runs only where nobody timed out.)"""
    import torch
    cfg = S.load_config(base_settings__experiment=experiment, **over)
    n, T1, T2 = 256, 6000, 20
    env = make_env(S, cfg, n, "fp32", 11, auto_reset=False)
    pol = constant_policy(c)
    act = np_(pol.act(env.obs, eps=torch.zeros((n, 1), device=env.device)))
    assert np.all(act == act[0, 0])
    a = float(act[0, 0])                              # the fp32 action the kernel takes
    s_y, knots = host_draws(cfg, n, 1, seed=11)
    before = env.counters()
    ret, steps, term = (np_(x) for x in pol.rollout(env, T1, deterministic=True))
    first = steps.astype(int)
    ref_out = oracle_ref(O, cfg, np.full((int(first.max()) + (0 if 4 in kinds else T2), n), a), s_y, knots,
                         auto_reset=False)
    ref = episode_reference(ref_out["reward"], ref_out["done"], ref_out["term"], auto_reset=False)
    d = ref_out["done"].astype(bool)
    want_first = np.where(d.any(0), d.argmax(0) + 1, min(T1, d.shape[0]))
    assert np.array_equal(first, want_first) and np.all(term > 0)
    assert np.array_equal(term, ref_out["term"][first - 1, np.arange(n)])
    assert set(np.unique(term)) == kinds
    cols = np.arange(n)
    check_within(f"rollout {name} return_out", ret, ref["running"][first - 1, cols], ref["run32"][first - 1, cols])
    first_only = episode_reference(np.where(np.arange(d.shape[0])[:, None] < first, ref_out["reward"], 0.0),
                                   d & (np.arange(d.shape[0])[:, None] < first), ref_out["term"], auto_reset=False)
    check_counters(env.counters(), first_only, "fp32", before)
    if 4 in kinds:
        env.close()
        return
    before = env.counters()
    ret2, steps2, term2 = (np_(x) for x in pol.rollout(env, T2, deterministic=True))
    rows = np.arange(d.shape[0])[:, None]
    nxt = np.array([first[i] + np.argmax(d[first[i]:, i]) + 1 if d[first[i]:, i].any() else first[i] + T2
                    for i in range(n)])
    assert np.array_equal(first + steps2.astype(int), nxt)
    assert np.array_equal(term2, ref_out["term"][nxt - 1, cols])
    check_within(f"rollout {name} second call return_out", ret2, ref["running"][nxt - 1, cols], ref["run32"][nxt - 1, cols])
    second = episode_reference(np.where((rows >= first) & (rows < nxt), ref_out["reward"], 0.0),
                               d & (rows >= first) & (rows < nxt), ref_out["term"], auto_reset=False)
    # the second call's episodes carry the whole return since reset: rebuild them from the cumulative running sum
    second["returns"] = ref["running"][nxt - 1, cols][d[nxt - 1, cols]]
    second["bound32"] = ref["run32"][nxt - 1, cols][d[nxt - 1, cols]]
    x = second["returns"]
    second["counts"][6:] = [math.fsum(x), math.fsum(x * x)]
    check_counters(env.counters(), second, "fp32", before)
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 7. the collect kernel (and its recording instantiation)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("record", [False, True])
def test_collect_counters_match_oracle(S, O, record, tmp_path):
    """Three collect chunks of T steps: the ring holds every action taken (row i of step t at slot
    (base_slot + t N + i) mod mem_size), and replaying them through the oracle gives the counters after each chunk;
    episodes end on the last step of a chunk, and the next chunk continues the others."""
    import torch
    from sac_agent_b200.networks import ActorNetwork, TensorCorePolicy
    cfg = S.load_config(base_settings__experiment=6)
    n, T, chunks = 4096, 70, 3
    env = make_env(S, cfg, n, "fp32", 17)
    torch.manual_seed(4)
    actor = ActorNetwork(None, (11,), max_action=[1.0]).cuda()
    with torch.no_grad():   # mean action ~tanh(1) plus noise: the rudder breaks after ~10-20 steps, at scattered steps
        actor.mean.weight.zero_()
        actor.mean.bias.fill_(1.0)
    pol = TensorCorePolicy(actor, seed=5)
    mem = S.ReplayBuffer(T * n + 1000, (11,), 1, precision="fp32", device=0, as_torch=True)
    rec = S.DeviceRecorder(env, [0, 1, 4095], str(tmp_path), capacity=T) if record else None
    s_y, knots = host_draws(cfg, n, chunks * T + 1, seed=17)
    actions, fields = [], []
    for chunk in range(chunks):
        base = mem.mem_cntr % mem.mem_size
        pol.collect(env, mem, T, recorder=rec)
        slots = (base + np.arange(T)[:, None] * n + np.arange(n)[None, :]) % mem.mem_size
        acts = mem.gather(torch.from_numpy(slots.reshape(-1)), as_torch=True)[1]
        actions.append(np_(acts).reshape(T, n))
        fields.append(np_(env.get_field("episode_reward")))
        ref_out = oracle_ref(O, cfg, np.concatenate(actions), s_y, knots)
        ref = episode_reference(ref_out["reward"], ref_out["done"], ref_out["term"])
        check_counters(env.counters(), ref, "fp32")
        check_within(f"collect record={record} chunk {chunk} running return", fields[-1], ref["running"][-1],
                     ref["run32"][-1])
    assert ref_out["done"][T - 1::T].any()   # episodes end on the last step of a chunk
    assert ref["counts"][5] > n
    if rec is not None:
        rec.close()
    env.close(); mem.close()


# ---------------------------------------------------------------------------------------------------------------------
# 8. sharded handles: all_reduce_counters at world size 1 and 2, info_from_counters
# ---------------------------------------------------------------------------------------------------------------------
SHARD_N, SHARD_T, SHARD_SEED = 2048, 900, 6


def shard_inputs():
    cfg = pkg().load_config(base_settings__experiment=6)
    return cfg, uniform(np.random.default_rng(SHARD_SEED), SHARD_T, SHARD_N, 1.0)


def check_reduced(out, ref):
    """all_reduce_counters' dict against the reference: counts exact, return_mean / return_var = the mean and the
    population variance of the episode returns (fp64 handles)."""
    x = ref["returns"]
    n = len(x)
    mean = math.fsum(x) / n
    var = math.fsum((x - mean) ** 2) / n
    for k, name in enumerate(KINDS + ("episodes",)):
        assert out[name] == ref["counts"][k]
    tol_sum, tol_sq = sum_tolerances(ref, "fp64")
    tol_mean = tol_sum / n + U64 * abs(mean)
    tol_var = tol_sq / n + 2 * abs(mean) * tol_mean + tol_mean ** 2 + 4 * U64 * (math.fsum(x * x) / n + mean * mean)
    assert abs(out["return_mean"] - mean) <= tol_mean, (out["return_mean"], mean, tol_mean)
    assert abs(out["return_var"] - var) <= tol_var, (out["return_var"], var, tol_var)
    from sac_agent_b200.experiment import info_from_counters
    info = info_from_counters(out)
    assert abs(info["episode_reward"] - mean) <= tol_mean
    assert [info[k] for k in KINDS] == list(ref["counts"][:5])


def shard_reference(O, lo, hi):
    cfg, a = shard_inputs()
    s_y, knots = host_draws(cfg, hi - lo, 12, seed=SHARD_SEED, env_id_offset=lo)
    r = oracle_ref(O, cfg, a[:, lo:hi], s_y, knots)
    return episode_reference(r["reward"], r["done"], r["term"])


@pytest.fixture
def gloo_world_1(tmp_path):
    """A one-rank gloo default group (file-store rendezvous), destroyed after the test."""
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/store", rank=0, world_size=1)
    yield
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_counters_world_1(S, O, gloo_world_1):
    """Two handles with env_id_offset; each shard's all_reduce_counters at world size 1 and the handles' summed
    counter vectors against the oracle."""
    import torch
    from sac_agent_b200.sharding import all_reduce_counters
    cfg, a = shard_inputs()
    half = SHARD_N // 2
    refs, tensors = [], []
    for lo, hi in ((0, half), (half, SHARD_N)):
        env = make_env(S, cfg, hi - lo, "fp64", SHARD_SEED, env_id_offset=lo)
        drive(env, a[:, lo:hi])
        refs.append(shard_reference(O, lo, hi))
        tensors.append(env.counters_tensor())
        check_reduced(all_reduce_counters(tensors[-1].clone()), refs[-1])
        env.close()
    check_reduced(all_reduce_counters(torch.stack(tensors).sum(0)), merge(*refs))


_WORKER = r"""
import json, os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch, torch.distributed as dist
import sac_agent_b200 as S
import test_episode_statistics as T
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
out_dir = sys.argv[1]
dist.init_process_group("gloo", init_method="file://" + out_dir + "/store", rank=rank, world_size=world)
cfg, a = T.shard_inputs()
lo, n = S.sharding.shard_range(T.SHARD_N, rank, world)
env = T.make_env(S, cfg, n, "fp64", T.SHARD_SEED, env_id_offset=lo)
T.drive(env, a[:, lo:lo + n])
out = S.sharding.all_reduce_counters(env.counters_tensor())
with open(os.path.join(out_dir, f"rank{{rank}}.json"), "w") as f:
    json.dump(out, f)
dist.barrier()
env.close()
dist.destroy_process_group()
print("SHARD_OK")
"""


@pytest.mark.gpu
def test_sharded_counters_two_ranks_over_gloo(S, O, tmp_path):
    """Two ranks (one process each, sharing cuda:0) own halves of the population; after all_reduce_counters both
    hold the statistics of all the envs' episodes."""
    script = tmp_path / "shard_worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK="0")
        procs.append(subprocess.Popen([sys.executable, str(script), str(tmp_path)], env=env, cwd=str(tmp_path),
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    for p in procs:
        out, err = p.communicate(timeout=600)
        assert p.returncode == 0 and "SHARD_OK" in out, err[-3000:]
    ranges = [S.shard_range(SHARD_N, r, 2) for r in range(2)]
    ref = merge(*(shard_reference(O, lo, lo + n) for lo, n in ranges))
    for r in range(2):
        check_reduced(json.loads((tmp_path / f"rank{r}.json").read_text()), ref)


# ---------------------------------------------------------------------------------------------------------------------
# 9. masked reset of live envs; state-dict round trip in mid-episode
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_masked_reset_and_resume_keep_the_statistics(S, O):
    """reset(mask) of running envs ends no episode and zeroes their running return (boat_env.py:122); a handle
    restored from a mid-episode state dict continues the counters and the running returns exactly."""
    import torch
    cfg = S.load_config(base_settings__experiment=6)
    n, T, T1, T2, E = 1024, 700, 200, 450, 12
    a = uniform(np.random.default_rng(12), T, n, 1.0)
    s_y, knots = host_draws(cfg, n, E + 1, seed=12)
    full = oracle_ref(O, cfg, a, s_y, knots)
    mask = np.arange(n) % 5 == 0
    # the masked envs: their steps up to T1, then a new episode with the next episode's draws
    ended = full["done"][:T1].sum(0).astype(int)
    live = mask & ~full["done"][T1 - 1].astype(bool)
    assert live.sum() > 150                             # the reset hits running episodes
    m = np.flatnonzero(mask)
    idx = ended[m][None, :] + 1 + np.arange(E - ended[m].max() - 1)[:, None]
    part2 = oracle_ref(O, cfg, a[T1:, m], s_y[idx, m], knots[idx, m])
    rew, dn, tm = full["reward"].copy(), full["done"].copy(), full["term"].copy()
    rew[T1:, m], dn[T1:, m], tm[T1:, m] = part2["reward"], part2["done"], part2["term"]
    restart = np.zeros((T, n), bool)
    restart[T1, m] = True
    ref = episode_reference(rew, dn, tm, restart=restart)
    env = make_env(S, cfg, n, "fp64", 12)
    done1, _ = drive(env, a[:T1])
    before = env.counters()
    env.reset(torch.from_numpy(mask).to(env.device))
    assert env.counters() == before                     # no episode counted
    rr = np_(env.get_field("episode_reward"))
    assert np.all(rr[mask] == 0.0)
    assert np.array_equal(np_(env.get_field("episode"))[mask], ended[mask] + 1)
    done2, field2 = drive(env, a[T1:T2])
    sd = env.state_dict()
    env.close()
    twin = S.BatchedBoatEnv(cfg, n, seed=12, precision="fp64", device=0, auto_reset=True)
    twin.load_state_dict(sd)
    check_within("masked reset running return before the checkpoint", np_(twin.get_field("episode_reward")),
                 ref["running"][T2 - 1], ref["run64"][T2 - 1])
    done3, field3 = drive(twin, a[T2:])
    assert np.array_equal(np.concatenate([done1, done2, done3]), dn)
    check_counters(twin.counters(), ref, "fp64")
    check_within("masked reset / resume running return", np.concatenate([field2, field3]), ref["running"][T1:],
                 ref["run64"][T1:])
    twin.close()


# ---------------------------------------------------------------------------------------------------------------------
# 10. all 32 counter rows under contention
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_counters_under_contention(S, O):
    """32768 envs (1024 state blocks, 32 per counter row), fp32, uniform actions of scale 4: the rudder breaks about
    every 28 steps, ~1.2 10^5 episodes in 100 steps."""
    cfg = S.load_config(base_settings__experiment=6)
    n, T = 32768, 100
    a = uniform(np.random.default_rng(10), T, n, 4.0)
    s_y, knots = host_draws(cfg, n, T // 3 + 2, seed=10)   # |a| <= 4: the rudder needs >= 3 steps to pass pi/3
    ref_out = oracle_ref(O, cfg, a, s_y, knots, n_threads=os.cpu_count() or 1)
    env = make_env(S, cfg, n, "fp32", 10)
    done, field = drive(env, a)
    ref = check_run(S, env, ref_out, done, field, "fp32", "contention")
    assert ref["counts"][5] > 100_000
    env.close()
