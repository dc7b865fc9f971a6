"""Population training on one GPU (population.AgentPopulation, boatagent_sac_update_members,
boatreplay_sample_members): the batched launches against the per-agent ones, bit for bit, and the host logic of
population rounds and of train_sac --population."""
import ctypes as C
import io
import math
import os
import random
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))

import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200 import _lib  # noqa: E402
from sac_agent_b200 import population as POP  # noqa: E402

EINVAL = -1
gpu = pytest.mark.gpu


# ---- CPU ------------------------------------------------------------------------------------------------------------

class _FakeMember:
    """What exploit_explore_local uses of a ContinuousAgent, on the CPU."""

    def __init__(self, k):
        self.t = [torch.full((3,), float(k)), torch.tensor([k, 10 * k], dtype=torch.int64)]
        self.hp = {"alpha": 1e-3, "beta": 1e-3 * (k + 1), "gamma": 0.99, "tau": 0.005}
        self.changed = 0

    def training_tensors(self):
        return self.t

    def hyperparameters(self):
        return dict(self.hp)

    def set_hyperparameters(self, **hp):
        self.hp = dict(hp)

    def _weights_changed(self):
        self.changed += 1


@pytest.mark.parametrize("scores, best, losers", [
    ([1.0, 2.0, 3.0, 4.0], 3, [0]),
    ([float("nan"), 2.0, 3.0, 3.0], 2, [0]),                        # NaN ranks last; the tie goes to the lower index
    ([5.0, 5.0, 5.0, 5.0], 0, []),                                   # nobody is worse than the best
    ([float("nan")] * 4, 0, []),                                     # no scores: no round
    ([1.0, 0.0, 7.0, float("nan"), 2.0, 3.0, 4.0, -1.0], 2, [3, 7]),   # bottom quarter of 8
])
def test_exploit_explore_local_decisions(scores, best, losers):
    members = [_FakeMember(k) for k in range(len(scores))]
    rng, ref_rng = random.Random(7), random.Random(7)
    info = POP.exploit_explore_local(members, scores, rng)
    assert info["best"] == best
    assert sorted(info["adopted"]) == sorted(losers)
    assert info["ranking"][0] == best and sorted(info["ranking"]) == list(range(len(scores)))
    best_hp = _FakeMember(best).hp
    for r in info["ranking"][len(scores) - len(losers):]:   # losers adopt in ranking order, one perturb draw each
        if r in losers:
            assert info["adopted"][r] == POP.perturb(best_hp, ref_rng)
    for k, m in enumerate(members):
        if k in losers:
            assert all(torch.equal(a, b) for a, b in zip(m.t, _FakeMember(best).t))
            assert m.hp == info["adopted"][k] and m.changed == 1
        else:
            assert all(torch.equal(a, b) for a, b in zip(m.t, _FakeMember(k).t)) and m.changed == 0
    # the ranking is the one exploit_explore uses
    assert POP.select([-float("inf") if math.isnan(s) else s for s in scores])[:2] == (info["ranking"], best)


def test_exploit_explore_local_rejects_a_short_score_table():
    with pytest.raises(ValueError):
        POP.exploit_explore_local([_FakeMember(0), _FakeMember(1)], [1.0], random.Random(0))


@pytest.mark.parametrize("flags", [
    ["--population", "4", "--data-parallel"],
    ["--population", "4", "--overlap"],
    ["--population", "4", "--record-envs", "4", "--experiments-root", "/nonexistent"],
    ["--population", "-1"],
    ["--population", "17"],
    ["--population", "4", "--learner-precision", "fp32"],          # an fp32 learner
    ["--population", "4", "--policy-precision", "fp32"],
    ["--population", "4", "--collect-steps", "0"],
])
def test_train_sac_population_rejects_before_cuda_work(flags, monkeypatch):
    import train_sac
    base = ["--policy-precision", "tcgen05", "--learner-precision", "tcgen05", "--collect-steps", "8"]
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("CUDA work before the flags were checked"))
    with pytest.raises(SystemExit):
        train_sac.main(base + flags)


def test_train_sac_population_rejects_cross_rank_rounds(monkeypatch):
    import train_sac
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("CUDA work before the flags were checked"))
    with pytest.raises(SystemExit):
        train_sac.main(["--policy-precision", "tcgen05", "--learner-precision", "tcgen05", "--collect-steps", "8",
                        "--population", "2", "--pbt-every", "5"])


def test_member_abi_rejects_bad_arguments_without_launching():
    L = S.lib()
    tbl = (_lib.SacMember * 17)()
    ws = C.c_void_p(16)
    for n in (0, 17, -1):
        assert L.boatagent_sac_update_members(tbl, n, 1024, 0.9, 0.999, 1e-8, ws, 1 << 40, None) == EINVAL
    assert L.boatagent_sac_update_members(None, 1, 1024, 0.9, 0.999, 1e-8, ws, 1 << 40, None) == EINVAL
    assert L.boatagent_sac_update_members(tbl, 1, 1000, 0.9, 0.999, 1e-8, ws, 1 << 40, None) == EINVAL   # batch % 128
    assert L.boatagent_sac_update_members(tbl, 1, 1024, 0.9, 0.999, 1e-8, ws, 1 << 40, None) == EINVAL   # NULL members
    smp = (_lib.SampleMember * 17)()
    for n in (0, 17):
        assert L.boatreplay_sample_members(smp, n, 1024, None) == EINVAL
    assert L.boatreplay_sample_members(None, 1, 1024, None) == EINVAL
    assert L.boatreplay_sample_members(smp, 1, 1024, None) == EINVAL    # NULL ring
    assert L.boatreplay_sample_members(smp, 1, 0, None) == EINVAL


# ---- GPU helpers ----------------------------------------------------------------------------------------------------

def _learner(seed):
    from sac_agent_b200.continuous_agent import SACLearner
    torch.manual_seed(seed)
    return SACLearner((11,), 1, np.ones(1, dtype=np.float32), 3e-4, 3e-4, 0.99, 0.005, 10.0, device="cuda")


def _set_hp(L, k):
    o = L.optimizer
    for i in range(len(o.params)):
        o._slots[i].lr = (3e-4 if i < 8 else 5e-4) * (1.0 + 0.37 * k)
    L.gamma = 0.99 - 0.01 * k
    L.tau = o.tau = 0.005 * (1 + k)
    L.scale = 10.0 + k


def _inputs(B, k):
    g = torch.Generator(device="cuda").manual_seed(1000 + k)
    kw = dict(device="cuda", generator=g)
    return (torch.rand((B, 11), **kw), torch.rand((B, 1), **kw) * 2 - 1, torch.randn(B, **kw),
            torch.rand((B, 11), **kw), (torch.rand(B, **kw) < 0.1).to(torch.uint8), torch.randn((2, B, 1), **kw))


def _bind(L):
    o = L.optimizer
    for i, p in enumerate(o.params):
        if p.grad is None:
            p.grad = torch.zeros_like(p)
        o._slots[i].grad = p.grad.data_ptr()
    return o


def _snapshot(L, losses):
    o = L.optimizer
    return ([p.detach().clone() for net in L.networks() for p in net.parameters()]
            + [p.grad.clone() for p in o.params] + [t.clone() for t in o.state_tensors()] + [losses.clone()])


def _assert_same(a, b, what):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), f"{what}: tensor {i} differs"


def _solo(L, inp, losses, ws):
    o = _bind(L)
    s, a, r, s2, d, eps = inp
    _lib.check(o._L.boatagent_sac_update(
        s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), eps.data_ptr(),
        L.actor.max_action.data_ptr(), s.shape[0], float(L.gamma), float(L.scale), o._slots, len(o.params),
        o.betas[0], o.betas[1], o.eps, o.tau, o.state.data_ptr(), losses.data_ptr(), ws.data_ptr(), ws.numel(), None),
        "boatagent_sac_update")


def _member(L, inp, losses):
    o = _bind(L)
    s, a, r, s2, d, eps = inp
    return _lib.SacMember(s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), eps.data_ptr(),
                          L.actor.max_action.data_ptr(), C.cast(o._slots, C.c_void_p), len(o.params), float(L.gamma),
                          float(L.scale), float(o.tau), o.state.data_ptr(), losses.data_ptr())


def _batched(Ls, inps, losses, ws, batch):
    tbl = (_lib.SacMember * len(Ls))(*[_member(L, i, l) for L, i, l in zip(Ls, inps, losses)])
    o = Ls[0].optimizer
    return o._L.boatagent_sac_update_members(tbl, len(Ls), batch, o.betas[0], o.betas[1], o.eps, ws.data_ptr(),
                                             ws.numel(), None)


# ---- GPU: the batched update ----------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("P", [1, 3, 5, 16])
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_batched_update_equals_solo_updates(P, B):
    solo = [_learner(10 + k) for k in range(P)]
    batch = [_learner(10 + k) for k in range(P)]
    for k in range(P):
        _set_hp(solo[k], k)
        _set_hp(batch[k], k)
    slice_bytes = int(S.lib().boatagent_sac_update_workspace_bytes(B))
    ws_solo = torch.empty(slice_bytes, dtype=torch.uint8, device="cuda")
    ws = torch.empty(P * slice_bytes, dtype=torch.uint8, device="cuda")
    l_solo = [torch.zeros(3, device="cuda") for _ in range(P)]
    l_batch = [torch.zeros(3, device="cuda") for _ in range(P)]
    for rnd in range(3):
        inps = [_inputs(B, 100 * rnd + k) for k in range(P)]
        for k in range(P):
            _solo(solo[k], inps[k], l_solo[k], ws_solo)
        assert _batched(batch, inps, l_batch, ws, B) == 0
        torch.cuda.synchronize()
        for k in range(P):
            _assert_same(_snapshot(solo[k], l_solo[k]), _snapshot(batch[k], l_batch[k]), f"round {rnd} member {k}")
        assert int(batch[0].optimizer.state[0]) == rnd + 1 and int(batch[-1].optimizer.state[1]) == 0
    if P > 1:   # the members really are different agents
        assert not torch.equal(batch[0].actor.fc2.weight, batch[1].actor.fc2.weight)


@gpu
def test_batched_update_rejections():
    B = 256
    Ls = [_learner(k) for k in range(2)]
    slice_bytes = int(S.lib().boatagent_sac_update_workspace_bytes(B))
    ws = torch.empty(2 * slice_bytes, dtype=torch.uint8, device="cuda")
    losses = [torch.zeros(3, device="cuda") for _ in range(2)]
    inps = [_inputs(B, k) for k in range(2)]
    tbl = (_lib.SacMember * 2)(*[_member(L, i, l) for L, i, l in zip(Ls, inps, losses)])   # binds the gradients
    before = _snapshot(Ls[1], losses[1])
    o = Ls[0].optimizer
    call = lambda t, n=2, b=B, nbytes=ws.numel(): o._L.boatagent_sac_update_members(  # noqa: E731
        t, n, b, 0.9, 0.999, 1e-8, ws.data_ptr(), nbytes, None)
    assert call(tbl, n=0) == EINVAL and call(tbl, n=17) == EINVAL
    assert call(tbl, nbytes=2 * slice_bytes - 1) == EINVAL                 # workspace too small
    assert call(tbl, b=B + 128, nbytes=ws.numel()) == EINVAL                # the shared batch needs a larger workspace
    Ls[1].optimizer._slots[2].numel -= 1                                    # a wrong slot numel (member 1)
    assert call(tbl) == EINVAL
    Ls[1].optimizer._slots[2].numel += 1
    tbl[1].n_slots = 25
    assert call(tbl) == EINVAL
    tbl[1].n_slots = 26
    tbl[1].adam_state = None
    assert call(tbl) == EINVAL
    torch.cuda.synchronize()
    _assert_same(before, _snapshot(Ls[1], losses[1]), "a rejected call changes nothing")


# ---- GPU: the batched gather ----------------------------------------------------------------------------------------

@gpu
def test_batched_gather_equals_solo_gathers():
    B = 1024
    specs = [(1000, 2500), (4096, B), (5000, 3000), (300_000, 200_000), (2048, 2048 * 3 + 17)]   # (size, rows stored)
    rings = []
    for k, (size, n) in enumerate(specs):
        r = S.ReplayBuffer(size, (11,), 1, precision="fp32", device=0, seed=77 + k, as_torch=True)
        g = torch.Generator(device="cuda").manual_seed(k)
        r.store_batch(torch.randn((n, 11), device="cuda", generator=g), torch.randn((n, 1), device="cuda", generator=g),
                      torch.randn(n, device="cuda", generator=g), torch.randn((n, 11), device="cuda", generator=g),
                      torch.rand(n, device="cuda", generator=g) < 0.3)
        r._samples = 3 * k
        rings.append(r)
    P = len(rings)
    for rnd in range(2):
        outs = [r._outputs(B) for r in rings]
        tbl = (_lib.SampleMember * P)(*[_lib.SampleMember(r._h, r.seed, r._samples, *[t.data_ptr() for t in o])
                                        for r, o in zip(rings, outs)])
        assert S.lib().boatreplay_sample_members(tbl, P, B, None) == 0
        for r, o in zip(rings, outs):
            ref = r.sample_buffer(B, as_torch=True, out=r._outputs(B))
            for x, y in zip(o, ref):
                assert torch.equal(x, y)
    assert [r._samples for r in rings] == [3 * k + 2 for k in range(P)]
    empty = S.ReplayBuffer(1000, (11,), 1, precision="fp32", device=0, as_torch=True)
    o = empty._outputs(B)
    tbl = (_lib.SampleMember * 1)(_lib.SampleMember(empty._h, 0, 0, *[t.data_ptr() for t in o]))
    assert S.lib().boatreplay_sample_members(tbl, 1, B, None) == -6   # BOATENV_ESTATE, as boatreplay_sample


# ---- GPU: the population --------------------------------------------------------------------------------------------

def _cfg(**kw):
    return S.load_config(base_settings__experiment=5, **kw)


def _agent_state(a):
    o = a.learner.optimizer
    return ([p.detach().clone() for net in a.learner.networks() for p in net.parameters()]
            + [p.grad.clone() for p in o.params] + [t.clone() for t in o.state_tensors()] + [a._loss_buf.clone()])


def _ring(a):
    sd = a.memory.state_dict()
    return [sd[k] for k in ("state", "action", "reward", "new_state", "terminal")], (sd["mem_cntr"], sd["samples"])


N_ENVS, T, U, BUF = 2048, 4, 3, 65536


@gpu
def test_population_of_one_is_todays_agent():
    seed, cfg = 3, _cfg()
    # the agent examples/train_sac.py builds at world 1
    torch.manual_seed(seed)
    env = S.make_sharded_env(cfg, N_ENVS, seed=seed, precision="fp32", auto_reset=True)
    mem = S.ReplayBuffer(BUF, (11,), 1, precision="fp32", device=0, seed=seed, as_torch=True)
    agent = S.ContinuousAgent(cfg, None, env.observation_space.shape, env, device=0, seed=seed, memory=mem,
                              policy_precision="tcgen05", learner_precision="tcgen05")
    env.reset()
    ref_losses = []
    for _ in range(5):
        agent.collect(env, T, done_flag_mode=1)
        for _ in range(U):
            out = agent.learn()
            if out is not None:
                ref_losses.append(torch.stack(out).clone())
    ref = (_agent_state(agent), _ring(agent), env.obs.clone(), env.counters(), agent.updates)

    torch.manual_seed(seed)
    pop = S.AgentPopulation(cfg, 1, N_ENVS, seed=seed, buffer_size=BUF)
    pop.reset()
    losses = []
    for _ in range(5):
        pop.collect(T)
        for _ in range(U):
            out = pop.learn()
            if out is not None:
                losses.append(torch.stack(out[0]).clone())
    a = pop.members[0]
    assert len(losses) == len(ref_losses) > 0
    _assert_same(ref_losses, losses, "losses")
    _assert_same(ref[0], _agent_state(a), "weights, gradients, Adam state")
    _assert_same(ref[1][0], _ring(a)[0], "ring")
    assert ref[1][1] == _ring(a)[1]
    assert torch.equal(ref[2], pop.envs[0].obs) and ref[3] == pop.envs[0].counters() and ref[4] == a.updates


def _solo_members(cfg, P, seed):
    """P ContinuousAgents built as AgentPopulation builds its members, each on its own."""
    from sac_agent_b200.networks import TensorCorePolicy
    out = []
    for g in range(P):
        env = S.BatchedBoatEnv(cfg, N_ENVS, seed=seed, precision="fp32", device=0, env_id_offset=g * N_ENVS)
        mem = S.ReplayBuffer(BUF, (11,), 1, precision="fp32", device=0, seed=seed + g, as_torch=True)
        torch.manual_seed(seed + g)
        a = S.ContinuousAgent(cfg, None, env.observation_space.shape, env, device=0, seed=seed + g, memory=mem,
                              policy_precision="tcgen05", learner_precision="tcgen05")
        a._tc_policy = TensorCorePolicy(a.actor, seed=0x5ac + g)
        env.reset()
        out.append((a, env))
    return out


@gpu
def test_population_loop_equals_independent_agents():
    seed, cfg, P = 11, _cfg(), 4
    pop = S.AgentPopulation(cfg, P, N_ENVS, seed=seed, buffer_size=BUF)
    pop.reset()
    solo = _solo_members(cfg, P, seed)
    n_learn = 0
    for _ in range(5):
        pop.collect(T)
        for a, env in solo:
            a.collect(env, T)
        for _ in range(U):
            out = pop.learn()
            if out is None:
                continue
            n_learn += 1
            for m, (a, env) in enumerate(solo):
                s, act, r, s2, d = a.memory.sample_buffer(a.batch_size, as_torch=True, out=a._batch)
                a.learn_from(s, act, r, s2, d, eps=pop.eps[m])
    torch.cuda.synchronize()
    assert n_learn > 0
    for m, (a, env) in enumerate(solo):
        b = pop.members[m]
        _assert_same(_agent_state(a), _agent_state(b), f"member {m}")
        _assert_same(_ring(a)[0], _ring(b)[0], f"ring {m}")
        assert _ring(a)[1] == _ring(b)[1] and torch.equal(env.obs, pop.envs[m].obs)
    # the members differ: weights, acting noise and wind draws
    assert not torch.equal(pop.members[0].actor.fc1.weight, pop.members[1].actor.fc1.weight)
    assert not torch.equal(pop.envs[0].obs, pop.envs[1].obs)
    assert pop.members[0]._tc_policy.seed != pop.members[1]._tc_policy.seed
    assert pop.envs[1].env_id_offset == N_ENVS


def _check_next_update_against_solo(pop):
    """One pop.learn() equals each member's own boatagent_sac_update on the same batch and draws."""
    before = [_agent_state(a) for a in pop.members]
    assert pop.learn() is not None
    torch.cuda.synchronize()
    after = [_agent_state(a) for a in pop.members]
    for a, st in zip(pop.members, before):
        with torch.no_grad():
            torch._foreach_copy_(_live(a), st)
        a._fused_update()   # the member's batch and draws are still in a._batch and a._eps
    torch.cuda.synchronize()
    for m, a in enumerate(pop.members):
        _assert_same(after[m], _agent_state(a), f"member {m}")


def _live(a):
    o = a.learner.optimizer
    return ([p.data for net in a.learner.networks() for p in net.parameters()] + [p.grad for p in o.params]
            + o.state_tensors() + [a._loss_buf])


@gpu
def test_population_round_and_new_hyperparameters():
    pop = S.AgentPopulation(_cfg(), 4, N_ENVS, seed=5, buffer_size=BUF)
    pop.reset()
    for _ in range(3):
        pop.collect(T)
        for _ in range(U):
            pop.learn()
    best_state = [t.clone() for t in pop.members[2].training_tensors()]
    best_hp = pop.members[2].hyperparameters()
    info = pop.exploit_explore([1.0, float("nan"), 5.0, 2.0], random.Random(3))
    assert info["best"] == 2 and list(info["adopted"]) == [1]
    hp = POP.perturb(best_hp, random.Random(3))
    assert info["adopted"][1] == hp
    _assert_same(best_state, [t.clone() for t in pop.members[1].training_tensors()], "adopted state")
    got = pop.members[1].hyperparameters()
    assert all(abs(got[k] - hp[k]) <= 1e-7 * max(1.0, abs(hp[k])) for k in hp)   # lr held as float32
    assert pop.members[1].learner.gamma == hp["gamma"] and pop.members[1].learner.tau == hp["tau"]
    _check_next_update_against_solo(pop)
    pop.set_hyperparameters(0, alpha=1e-3, gamma=0.95, tau=0.02)
    _check_next_update_against_solo(pop)


@gpu
def test_population_checkpoint_and_resume():
    pop = S.AgentPopulation(_cfg(), 3, N_ENVS, seed=9, buffer_size=BUF)
    pop.reset()
    for _ in range(3):
        pop.collect(T)
        for _ in range(U):
            pop.learn()
    buf = io.BytesIO()
    torch.save(pop.state_dict(), buf)

    def run_on():
        out = []
        for _ in range(4):
            out += [torch.stack(l).clone() for l in pop.learn()]
        torch.cuda.synchronize()
        return out + [t for a in pop.members for t in _agent_state(a)]

    first = run_on()
    buf.seek(0)
    pop.load_state_dict(torch.load(buf, weights_only=False))
    _assert_same(first, run_on(), "resumed run")


@gpu
def test_population_rejections():
    with pytest.raises(ValueError):
        S.AgentPopulation(_cfg(), 17, 256)
    with pytest.raises(ValueError):
        S.AgentPopulation(_cfg(), 0, 256)
    with pytest.raises(ValueError):   # mismatched batch sizes
        S.AgentPopulation(_cfg(), 2, 256, configs=[_cfg(), _cfg(agent__batch_size=512)], buffer_size=4096)
