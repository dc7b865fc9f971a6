"""SAC-v2 (SAC2Learner, ContinuousAgent(algorithm="sac2"), boatagent_sac2_update_members): the PyTorch learner against
an independent float64 restatement of the update, a bf16 emulation of the fused kernels anchored to that learner, the
ABI's and the drivers' rejections, and on the GPU the fp32 graph, the fused update, populations, checkpoints and the
drivers end to end.

The update (alpha = exp(log_alpha) before the update, every loss on the weights before it, then one Adam step over
three learning rates and the Polyak average of both target critics):
  y = scale r + gamma (1 - done) (min(Qt1, Qt2)(s', a') - alpha lp'),   a', lp' = actor.sample_normal(s', eps[0])
  critic_loss = 0.5 mse(Q1(s, a), y) + 0.5 mse(Q2(s, a), y)
  actor_loss = mean(alpha lp - min(Q1, Q2)(s, a~)),   a~, lp = actor.sample_normal(s, eps[1]), actor gradients only
  temperature_loss = -log_alpha mean(lp + target_entropy), lp detached
"""
import ctypes as C
import json
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200 import _lib  # noqa: E402
from sac_agent_b200.continuous_agent import ContinuousAgent, SAC2Learner, _AdamSlot  # noqa: E402
from test_gpu_learner import _env_stub, _gauss_bwd, _gauss_fwd  # noqa: E402

gpu = pytest.mark.gpu
EINVAL, EALIGN = -1, -7
CRITICS = ("critic_1", "critic_2")
TARGETS = ("target_critic_1", "target_critic_2")
NETS = ("actor",) + CRITICS + TARGETS
HEADS = {"actor": ("mean", "std"), "critic_1": ("q",), "critic_2": ("q",), "target_critic_1": ("q",),
         "target_critic_2": ("q",)}
TRAINED = ("actor",) + CRITICS


def _params(L, dtype=torch.float32):
    """{net: {name: tensor}} of the five networks and log_alpha [1] (detached copies)."""
    P = {n: {k: p.detach().clone().to(dtype) for k, p in getattr(L, n).named_parameters()} for n in NETS}
    return P, L.temperature.log_alpha.detach().clone().to(dtype)


def _batch(B, seed, device="cpu"):
    g = torch.Generator(device="cpu").manual_seed(seed)
    st = torch.rand(B, 11, generator=g) * 2 - 1
    done = torch.rand(B, generator=g) < 0.2
    done[:3] = True
    out = dict(state=st, action=torch.rand(B, 1, generator=g) * 2 - 1, reward=torch.randn(B, generator=g),
               new_state=st + 0.1 * torch.randn(B, 11, generator=g), done=done, eps=torch.randn(2, B, 1, generator=g))
    return {k: v.to(device) for k, v in out.items()}


def _perturb(L, scale=0.02, seed=0):
    """Weights away from the initialisation, and target critics that are not the critics."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    with torch.no_grad():
        for net in (L.actor, L.critic_1, L.critic_2, L.target_critic_1, L.target_critic_2):
            for p in net.parameters():
                p.add_((scale * torch.randn(p.shape, generator=g)).to(p.device))
        L.temperature.log_alpha.fill_(math.log(0.3))


def _tie_critics(L):
    """Critic 2 (and its target) := critic 1: every min(Q1, Q2) is a tie."""
    with torch.no_grad():
        for a, b in ((L.critic_1, L.critic_2), (L.target_critic_1, L.target_critic_2)):
            for p, q in zip(a.parameters(), b.parameters()):
                q.copy_(p)


# ---- the float64 restatement --------------------------------------------------------------------------------------

def restate_f64(P, log_alpha, b, gamma, scale, target_entropy, max_action=1.0):
    """The update written out in float64 with autograd.  Returns ({net: {name: grad}} with "log_alpha", [3] losses)."""
    W = {n: {k: v.double().clone().requires_grad_(True) for k, v in P[n].items()} for n in NETS}
    la = log_alpha.double().clone().requires_grad_(True)
    s, a, r, s2 = (b[k].double() for k in ("state", "action", "reward", "new_state"))
    done, e = b["done"].double(), b["eps"].double().reshape(2, -1, 1)

    def mlp(n, x):
        w = W[n]
        h = torch.relu(x @ w["fc1.weight"].T + w["fc1.bias"])
        h = torch.relu(h @ w["fc2.weight"].T + w["fc2.bias"])
        return [h @ w[f"{k}.weight"].T + w[f"{k}.bias"] for k in HEADS[n]]

    def sample(x, eps):
        mean, raw = mlp("actor", x)
        log_std = -5.0 + 3.5 * (torch.tanh(raw) + 1.0)
        std = log_std.exp()
        u = mean + eps * std
        act = torch.tanh(u) * max_action
        lp = -((u - mean) ** 2) / (2 * std * std) - log_std - 0.5 * math.log(2 * math.pi)
        lp = lp - torch.log(1 - act ** 2 + 1e-6)
        return act, lp.sum(1)

    def q(n, x, act):
        return mlp(n, torch.cat([x, act], 1))[0].view(-1)

    with torch.no_grad():
        alpha = la.exp()
        a2, lp2 = sample(s2, e[0])
        y = scale * r + gamma * (1 - done) * (torch.min(q("target_critic_1", s2, a2), q("target_critic_2", s2, a2))
                                              - alpha * lp2)
    critic_loss = 0.5 * ((q("critic_1", s, a) - y) ** 2).mean() + 0.5 * ((q("critic_2", s, a) - y) ** 2).mean()
    cp = [W[n][k] for n in CRITICS for k in W[n]]
    gc = torch.autograd.grad(critic_loss, cp)
    at, lp = sample(s, e[1])
    actor_loss = (alpha.detach() * lp - torch.min(q("critic_1", s, at), q("critic_2", s, at))).mean()
    ap = list(W["actor"].values())
    ga = torch.autograd.grad(actor_loss, ap)
    temperature_loss = -(la * (lp.detach() + target_entropy).mean()).sum()
    gt = torch.autograd.grad(temperature_loss, [la])
    grads = {"actor": dict(zip(W["actor"], ga)), "log_alpha": gt[0]}
    i = 0
    for n in CRITICS:
        grads[n] = {}
        for k in W[n]:
            grads[n][k] = gc[i]
            i += 1
    return grads, torch.stack([temperature_loss.detach(), actor_loss.detach(), critic_loss.detach()])


def _reference(seed=0):
    torch.manual_seed(seed)
    return SAC2Learner((11,), 1, np.ones(1, dtype=np.float32), 5e-3, 3e-4, 0.99, 0.005, 10.0, device="cpu",
                       torch_reference_math=True, temperature_lr=7e-4)


def _grads_of(L):
    out = {n: {k: p.grad for k, p in getattr(L, n).named_parameters()} for n in TRAINED}
    out["log_alpha"] = L.temperature.log_alpha.grad
    return out


def _assert_grads(got, ref, rel):
    worst = {}
    for n in TRAINED:
        for k, r in ref[n].items():
            err = (got[n][k].double() - r.double()).abs().max().item() / max(r.abs().max().item(), 1e-30)
            worst[f"{n}.{k}"] = err
    r = ref["log_alpha"]
    worst["log_alpha"] = (got["log_alpha"].double() - r.double()).abs().max().item() / max(r.abs().max().item(), 1e-30)
    bad = {k: v for k, v in worst.items() if v > rel}
    assert not bad, bad
    return worst


@pytest.mark.parametrize("tied", [False, True])
def test_reference_learner_is_the_float64_restatement(tied):
    L = _reference(1)
    _perturb(L, seed=2)
    if tied:
        _tie_critics(L)
    b = _batch(256, 3)
    P, la = _params(L)
    ref_g, ref_l = restate_f64(P, la, b, L.gamma, L.scale, L.target_entropy)
    losses = L.update(b["state"], b["action"], b["reward"], b["new_state"], b["done"], eps_sample=b["eps"][0],
                      eps_rsample=b["eps"][1])
    _assert_grads(_grads_of(L), ref_g, 1e-5)
    assert torch.allclose(torch.stack(list(losses)).double(), ref_l, rtol=1e-5, atol=1e-6), (losses, ref_l)

    # the step: torch.optim.Adam over the three groups, and a hand Polyak average into both target critics
    params = [P["actor"][k].clone().requires_grad_(True) for k in P["actor"]]
    crit = [P[n][k].clone().requires_grad_(True) for n in CRITICS for k in P[n]]
    la_p = la.clone().requires_grad_(True)
    grads = _grads_of(L)
    for p, g in zip(params + crit + [la_p], [grads["actor"][k] for k in P["actor"]] +
                    [grads[n][k] for n in CRITICS for k in P[n]] + [grads["log_alpha"]]):
        p.grad = g.clone()
    opt = torch.optim.Adam([{"params": params, "lr": 5e-3}, {"params": crit, "lr": 3e-4}, {"params": [la_p], "lr": 7e-4}])
    opt.step()
    assert all(torch.equal(p, q) for p, q in zip(params, L.actor.parameters()))
    assert all(torch.equal(p, q) for p, q in zip(crit, list(L.critic_1.parameters()) + list(L.critic_2.parameters())))
    assert torch.equal(la_p, L.temperature.log_alpha)
    old_t = [P[n][k] for n in TARGETS for k in P[n]]
    new_t = list(L.target_critic_1.parameters()) + list(L.target_critic_2.parameters())
    for c, t_old, t_new in zip(crit, old_t, new_t):
        assert torch.allclose(t_new, 0.005 * c.detach() + (1 - 0.005) * t_old, rtol=0, atol=1e-7)
    if tied:   # the tie split: both critics' Q at (s, a~) enter the actor's gradient with weight 1/2
        assert torch.equal(L.critic_1.fc2.weight, L.critic_2.fc2.weight)


def test_reference_learner_layout():
    L = _reference(0)
    assert [n.name for n in L.networks()] == ["actor_network", "critic_network_1", "critic_network_2",
                                              "target_critic_network_1", "target_critic_network_2", "log_alpha"]
    assert L.target_entropy == -1.0 and float(L.alpha()) == pytest.approx(1.0)
    assert len(L.optimizer_params()) == 21 and L.optimizer_params()[-1] is L.temperature.log_alpha
    assert all(torch.equal(p, q) for p, q in zip(L.critic_1.parameters(), L.target_critic_1.parameters()))
    assert [g["lr"] for g in L.optimizer.param_groups] == [5e-3, 3e-4, 7e-4]
    torch.manual_seed(0)
    L2 = SAC2Learner((11,), 1, np.ones(1, dtype=np.float32), 5e-3, 3e-4, 0.99, 0.005, 10.0, device="cpu",
                     torch_reference_math=True, init_temperature=0.1, target_entropy=-2.0)
    assert float(L2.alpha()) == pytest.approx(0.1) and L2.target_entropy == -2.0
    assert [g["lr"] for g in L2.optimizer.param_groups] == [5e-3, 3e-4, 3e-4]   # temperature_lr defaults to beta
    assert all(torch.equal(p, q) for p, q in zip(L.actor.parameters(), L2.actor.parameters()))   # fixed creation order
    with pytest.raises(RuntimeError):
        SAC2Learner((11,), 1, np.ones(1, dtype=np.float32), 5e-3, 3e-4, 0.99, 0.005, 10.0, device="cpu")


# ---- the bf16 emulation of the fused kernels ----------------------------------------------------------------------

def emulate_update_sac2(P, log_alpha, b, gamma, scale, target_entropy, max_action=1.0, rounding=True):
    """One SAC-v2 update of the fused learner: bf16 rounding exactly where the kernels feed the tensor cores (fc1's
    inputs and weights, H1 into fc2, fc2's weights, dZ2 into dZ2 . W2 and dZ2^T . H1), everything else fp32.  Returns
    ({net: {name: grad}} with "log_alpha", [3] losses)."""
    r = (lambda t: t.to(torch.bfloat16).float()) if rounding else (lambda t: t)  # noqa: E731
    state, new_state, reward, done = b["state"], b["new_state"], b["reward"], b["done"]
    B = state.shape[0]
    a_b, e = b["action"].reshape(B), b["eps"].reshape(2, B)

    def fwd(n, x):
        p = P[n]
        h1 = torch.relu(r(x) @ r(p["fc1.weight"]).T + p["fc1.bias"])
        h1b = r(h1)
        h2 = torch.relu(h1b @ r(p["fc2.weight"]).T + p["fc2.bias"])
        return dict(x=x, h1=h1, h1b=h1b, h2=h2, y=[h2 @ p[h + ".weight"][0] + p[h + ".bias"][0] for h in HEADS[n]])

    def bwd(n, f, dys):
        p = P[n]
        dh2 = sum(dy[:, None] * p[h + ".weight"][0][None, :] for dy, h in zip(dys, HEADS[n]))
        dz2 = dh2 * (f["h2"] > 0)
        dz1 = (r(dz2) @ r(p["fc2.weight"])) * (f["h1"] > 0)
        g = {"fc1.weight": dz1.T @ f["x"], "fc1.bias": dz1.sum(0), "fc2.weight": r(dz2).T @ f["h1b"],
             "fc2.bias": dz2.sum(0)}
        for dy, h in zip(dys, HEADS[n]):
            g[h + ".weight"] = (dy[:, None] * f["h2"]).sum(0)[None]
            g[h + ".bias"] = dy.sum()[None]
        return g, dz1 @ p["fc1.weight"]

    alpha = torch.exp(log_alpha)[0]
    a_next, lp_next = _gauss_fwd(*fwd("actor", new_state)["y"], e[0], max_action)
    fa = fwd("actor", state)
    mean, raw = fa["y"]
    a_pi, lp = _gauss_fwd(mean, raw, e[1], max_action)
    qt = [fwd(t, torch.cat([new_state, a_next[:, None]], 1))["y"][0] for t in TARGETS]
    v_next = torch.minimum(qt[0], qt[1]) - alpha * lp_next
    q_hat = scale * reward + gamma * torch.where(done, torch.zeros_like(v_next), v_next)
    grads, q_pi, dq_pi, q_sa = {}, [], [], []
    for n in CRITICS:
        f2 = fwd(n, torch.cat([state, a_pi[:, None]], 1))
        q_pi.append(f2["y"][0])
        dq_pi.append(bwd(n, f2, [torch.ones_like(a_pi)])[1][:, -1])
        fs = fwd(n, torch.cat([state, a_b[:, None]], 1))
        q_sa.append(fs["y"][0])
        grads[n] = bwd(n, fs, [(fs["y"][0] - q_hat) / B])[0]

    def share(x, y):
        return torch.where(x < y, 1.0, torch.where(x == y, 0.5, 0.0))
    ga = -(share(q_pi[0], q_pi[1]) * dq_pi[0] + share(q_pi[1], q_pi[0]) * dq_pi[1]) / B
    gm, gr = _gauss_bwd(mean, raw, e[1], max_action, ga, torch.full_like(ga, 1.0 / B) * alpha)
    grads["actor"] = bwd("actor", fa, [gm, gr])[0]
    ent = (lp + target_entropy).mean()
    grads["log_alpha"] = -ent[None]
    losses = torch.stack([-log_alpha[0] * ent, (alpha * lp - torch.minimum(q_pi[0], q_pi[1])).mean(),
                          0.5 * ((q_sa[0] - q_hat) ** 2).mean() + 0.5 * ((q_sa[1] - q_hat) ** 2).mean()])
    return grads, losses


def test_emulation_without_rounding_is_the_reference_learner():
    L = _reference(4)
    _perturb(L, seed=5)
    b = _batch(384, 6)
    P, la = _params(L)
    grads, losses = emulate_update_sac2(P, la, b, L.gamma, L.scale, L.target_entropy, rounding=False)
    ref = L.update(b["state"], b["action"], b["reward"], b["new_state"], b["done"], eps_sample=b["eps"][0],
                   eps_rsample=b["eps"][1])
    _assert_grads(grads, _grads_of(L), 2e-5)
    assert torch.allclose(losses, torch.stack(list(ref)), rtol=1e-5, atol=1e-7)


# ---- ABI and argument rejections (no launch) ----------------------------------------------------------------------

def _fake_slots(n=21):
    """A host table of 21 well-formed slots with fake device addresses (only checked, never dereferenced)."""
    numel = [256 * 11, 256, 256 * 256, 256, 256, 1, 256, 1] + [256 * 12, 256, 256 * 256, 256, 256, 1] * 2 + [1]
    slots = (_AdamSlot * n)()
    for k in range(n):
        base = 0x10000000 * (k + 1)
        slots[k] = _AdamSlot(base, base + 0x1000000, base + 0x2000000, base + 0x3000000,
                             base + 0x4000000 if 8 <= k < 20 else None, numel[k] if k < 21 else 1, 1e-3, 0)
    return slots


def _fake_member(slots, n_slots=21):
    m = _lib.SacMember(*[0x1000 * (k + 1) for k in range(7)], C.cast(slots, C.c_void_p), n_slots, 0.99, 10.0, 0.005,
                       0x9000, 0xa000)
    return _lib.Sac2Member(m, -1.0)


def test_sac2_abi_rejects_bad_tables_without_launching():
    L = S.lib()
    ws, big = C.c_void_p(1 << 20), 1 << 40

    def call(tbl, n=1, batch=1024, ws_bytes=big, workspace=ws):
        return L.boatagent_sac2_update_members(tbl, n, batch, 0.9, 0.999, 1e-8, workspace, ws_bytes, None)

    assert L.boatagent_sac2_update_workspace_bytes(0) == EINVAL and L.boatagent_sac2_update_workspace_bytes(130) == EINVAL
    per = int(L.boatagent_sac2_update_workspace_bytes(1024))
    assert 0 < per < int(L.boatagent_sac_update_workspace_bytes(1024))   # three trained networks instead of four
    slots = _fake_slots()
    good = (_lib.Sac2Member * 17)(*[_fake_member(slots)] * 17)
    for n in (0, 17, -1):
        assert call(good, n) == EINVAL
    assert call(None) == EINVAL
    assert call((_lib.Sac2Member * 1)()) == EINVAL                      # NULL pointers
    for batch in (0, 1000, -128):
        assert call(good, batch=batch) == EINVAL
    assert call(good, workspace=None) == EINVAL
    assert call(good, ws_bytes=per - 1) == EINVAL                       # short workspace, one member
    assert call(good, 3, ws_bytes=3 * per - 16) == EINVAL               # short workspace, three members
    assert call(good, workspace=C.c_void_p((1 << 20) + 8)) == EALIGN
    for n_slots in (20, 26):
        assert call((_lib.Sac2Member * 1)(_fake_member(_fake_slots(26), n_slots))) == EINVAL

    def mutated(k, field, value):
        s = _fake_slots()
        setattr(s[k], field, value)
        return (_lib.Sac2Member * 2)(_fake_member(_fake_slots()), _fake_member(s))   # the bad entry is member 1

    assert call(mutated(8, "target", None), 2) == EINVAL                # a critic without its target
    assert call(mutated(19, "target", None), 2) == EINVAL
    assert call(mutated(0, "target", 0x5000), 2) == EINVAL              # an extra target on the actor
    assert call(mutated(20, "target", 0x5000), 2) == EINVAL             # ... and on log alpha
    assert call(mutated(20, "param", None), 2) == EINVAL                # a NULL log alpha
    assert call(mutated(20, "numel", 2), 2) == EINVAL
    assert call(mutated(2, "numel", 256 * 255), 2) == EINVAL
    assert call(mutated(5, "grad", None), 2) == EINVAL
    assert call(mutated(20, "param", 0x10000004), 2) == EALIGN
    m = _fake_member(slots)
    m.base.adam_state = None
    assert call((_lib.Sac2Member * 1)(m)) == EINVAL


@pytest.mark.parametrize("flags", [
    ["--algorithm", "sac2", "--data-parallel"],
    ["--algorithm", "sac2", "--overlap"],
    ["--algorithm", "sac2", "--population", "2", "--data-parallel", "--policy-precision", "tcgen05",
     "--learner-precision", "tcgen05", "--collect-steps", "4"],
    ["--algorithm", "sac2", "--init-temperature", "0"],
    ["--target-entropy", "-2"],                          # the temperature flags need --algorithm sac2
    ["--temperature-lr", "1e-3"],
    ["--init-temperature", "0.5"],
    ["--algorithm", "sac3"],
])
def test_train_sac_rejects_sac2_combinations_before_cuda_work(flags, monkeypatch):
    import train_sac
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("CUDA work before the flags were checked"))
    with pytest.raises(SystemExit):
        train_sac.main(flags)


def test_train_sac_rejects_sac2_rounds_across_ranks(monkeypatch):
    import train_sac
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("CUDA work before the flags were checked"))
    with pytest.raises(SystemExit):
        train_sac.main(["--algorithm", "sac2", "--pbt-every", "5"])


def test_agent_and_population_reject_sac2_combinations(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: pytest.fail("CUDA work before the arguments were checked"))
    cfg = S.load_config()
    for kw in ({"algorithm": "sac2", "data_parallel": True}, {"algorithm": "sac3"}, {"target_entropy": -2.0},
               {"temperature_lr": 1e-3}, {"init_temperature": 0.5}):
        with pytest.raises(ValueError):
            ContinuousAgent(cfg, None, (11,), _env_stub(), **kw)
    for kw in ({"algorithm": "sac2", "data_parallel": True}, {"algorithm": "sac3"}, {"target_entropy": -2.0}):
        with pytest.raises(ValueError):
            S.AgentPopulation(cfg, 2, 128, **kw)


# ---- GPU -----------------------------------------------------------------------------------------------------------

def _agent(batch, learner_precision="tcgen05", seed=0, **kw):
    cfg = S.load_config(agent__batch_size=batch)
    mem = kw.pop("memory", None) or S.ReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    torch.manual_seed(seed)
    return ContinuousAgent(cfg, None, (11,), _env_stub(), device=0, memory=mem, learner_precision=learner_precision,
                           algorithm="sac2", **kw)


def _learn(agent, b):
    return agent.learn_from(b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8),
                            eps=b["eps"])


def _snapshot(agent):
    L, o = agent.learner, agent.learner.optimizer
    return ([p.detach().clone() for net in L.networks() for p in net.parameters()] +
            [p.grad.clone() for p in o.params] + [t.clone() for t in o.state_tensors()])


def _adam_emulation(agent, P, log_alpha, grads):
    """What DeviceAdam's step makes of P and log_alpha with `grads` (fp32, three groups, Polyak into both targets)."""
    o = agent.learner.optimizer
    t = int(o.state[0]) + 1
    b1, b2 = o.betas
    bc1, bc2s = 1.0 - b1 ** t, (1.0 - b2 ** t) ** 0.5
    names = [(n, k) for n in TRAINED for k in P[n]] + [("log_alpha", None)]
    new = {n: dict(P[n]) for n in NETS}
    for i, (n, k) in enumerate(names):
        g = grads[n][k] if k else grads[n]
        m, v = o.exp_avg[i].float(), o.exp_avg_sq[i].float()
        m2 = m + (g - m) * (1 - b1)
        v2 = v * b2 + (1 - b2) * g * g
        x = (P[n][k] if k else log_alpha) - (o._slots[i].lr / bc1) * (m2 / (v2.sqrt() / bc2s + o.eps))
        if k is None:
            new["log_alpha"] = x
            continue
        new[n][k] = x
        if n in CRITICS:
            tn = TARGETS[CRITICS.index(n)]
            new[tn][k] = o.tau * x + (1 - o.tau) * P[tn][k]
    return new


def _check_update(agent, b, grad_tol=2e-3, loss_rtol=2e-3):
    """One fused learn_from against the emulation from the weights before it: every .grad within grad_tol of its
    tensor's largest gradient, the weights and targets within the lr-based tolerance of v1's check, the losses."""
    L = agent.learner
    P, la = _params(L)
    grads, losses = emulate_update_sac2(P, la, b, L.gamma, L.scale, L.target_entropy)
    expect = _adam_emulation(agent, P, la, grads)
    got_losses = _learn(agent, b)
    torch.cuda.synchronize()
    worst = _assert_grads(_grads_of(L), grads, grad_tol)
    for i, n in enumerate(TRAINED):
        lr = float(L.optimizer._slots[0 if n == "actor" else 8].lr)
        for k, p in getattr(L, n).named_parameters():
            werr = (p.detach() - expect[n][k]).abs()
            assert (werr > 1e-6 + 0.02 * lr).float().mean().item() <= 0.002, (n, k, werr.max().item())
    lr_t = float(L.optimizer._slots[20].lr)
    assert (L.temperature.log_alpha.detach() - expect["log_alpha"]).abs().item() <= 1e-6 + 0.02 * lr_t
    for tn in TARGETS:
        for k, p in getattr(L, tn).named_parameters():
            assert (p.detach() - expect[tn][k]).abs().max().item() <= 1e-6 + 0.02 * 3e-4 * L.tau + 1e-7, (tn, k)
    got = torch.stack([x.detach() for x in got_losses])
    assert torch.allclose(got, losses, rtol=loss_rtol, atol=1e-6), (got, losses)
    return worst


def _away_from_init(agent, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for p in agent.learner.optimizer_params()[:-1]:
            p.add_(0.02 * torch.randn(p.shape, device="cuda", generator=g))
        agent.learner.update_network_parameters(tau=1.0)


@gpu
def test_fp32_graph_update_is_the_eager_update_and_the_restatement():
    agents = [_agent(256, "fp32", seed=7, use_cuda_graph=g) for g in (True, False)]
    for a in agents:
        _away_from_init(a, 1)
    for u in range(3):
        b = _batch(256, 40 + u, "cuda")
        if u == 0:
            P, la = _params(agents[0].learner)
            ref_g, ref_l = restate_f64(P, la, b, agents[0].learner.gamma, agents[0].learner.scale, -1.0)
        ls = [_learn(a, b) for a in agents]
        torch.cuda.synchronize()
        assert all(torch.equal(x, y) for x, y in zip(ls[0], ls[1]))
        assert all(torch.equal(x, y) for x, y in zip(_snapshot(agents[0]), _snapshot(agents[1]))), u
        if u == 0:
            worst = _assert_grads(_grads_of(agents[0].learner), ref_g, 1e-4)
            print(f"fp32 graph vs float64: worst {max(worst.values()):.2e} ({max(worst, key=worst.get)})")
            assert torch.allclose(torch.stack(list(ls[0])).double(), ref_l, rtol=1e-4, atol=1e-5)
    assert int(agents[0].learner.optimizer.state[0]) == 3
    for a in agents:
        a.memory.close()


@gpu
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_fused_update_matches_emulation(B):
    agent = _agent(B, seed=B)
    _away_from_init(agent, B)
    with torch.no_grad():
        agent.learner.temperature.log_alpha.fill_(math.log(0.2))
    worst = {}
    for u in range(3):
        for k, v in _check_update(agent, _batch(B, 100 * B + u, "cuda")).items():
            worst[k] = max(worst.get(k, 0.0), v)
    print(f"sac2 B={B}: worst |grad - emulation| / max|grad| = {max(worst.values()):.2e} ({max(worst, key=worst.get)})")
    o = agent.learner.optimizer
    assert int(o.state[0]) == 3 and int(o.state[1]) == 0
    agent.memory.close()


@gpu
def test_fused_update_is_bit_reproducible():
    agents = [_agent(1024, seed=4) for _ in range(2)]
    agents[1].load_state_dict(agents[0].state_dict())
    for u in range(3):
        b = _batch(1024, u, "cuda")
        ls = [_learn(a, b) for a in agents]
        assert all(torch.equal(x, y) for x, y in zip(ls[0], ls[1]))
    assert all(torch.equal(x, y) for x, y in zip(_snapshot(agents[0]), _snapshot(agents[1])))
    for a in agents:
        a.memory.close()


def _gpu_learner(seed, k):
    torch.manual_seed(seed)
    L = SAC2Learner((11,), 1, np.ones(1, dtype=np.float32), 3e-4, 3e-4, 0.99, 0.005, 10.0, device="cuda",
                    target_entropy=-1.0 - 0.25 * k, init_temperature=0.5 + 0.1 * k, temperature_lr=1e-3 * (1 + 0.3 * k))
    o = L.optimizer
    for i in range(20):
        o._slots[i].lr = (3e-4 if i < 8 else 5e-4) * (1.0 + 0.37 * k)
    L.gamma, L.scale = 0.99 - 0.01 * k, 10.0 + k
    L.tau = o.tau = 0.005 * (1 + k)
    for i, p in enumerate(o.params):
        p.grad = torch.zeros_like(p)
        o._slots[i].grad = p.grad.data_ptr()
    return L


def _members(Ls, inps, losses):
    tbl = (_lib.Sac2Member * len(Ls))()
    for m, (L, inp, l) in enumerate(zip(Ls, inps, losses)):
        o = L.optimizer
        s, a, r, s2, d, eps = inp
        tbl[m] = _lib.Sac2Member(_lib.SacMember(
            s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), eps.data_ptr(),
            L.actor.max_action.data_ptr(), C.cast(o._slots, C.c_void_p), len(o.params), float(L.gamma), float(L.scale),
            float(o.tau), o.state.data_ptr(), l.data_ptr()), float(L.target_entropy))
    return tbl


def _inputs(B, k):
    g = torch.Generator(device="cuda").manual_seed(1000 + k)
    kw = dict(device="cuda", generator=g)
    return (torch.rand((B, 11), **kw), torch.rand((B, 1), **kw) * 2 - 1, torch.randn(B, **kw),
            torch.rand((B, 11), **kw), (torch.rand(B, **kw) < 0.1).to(torch.uint8), torch.randn((2, B, 1), **kw))


@gpu
@pytest.mark.parametrize("P", [1, 3, 16])
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_population_update_equals_solo_updates(P, B):
    Lib = S.lib()
    solo = [_gpu_learner(10 + k, k) for k in range(P)]
    pop = [_gpu_learner(10 + k, k) for k in range(P)]
    per = int(Lib.boatagent_sac2_update_workspace_bytes(B))
    ws_solo = torch.empty(per, dtype=torch.uint8, device="cuda")
    ws = torch.empty(P * per, dtype=torch.uint8, device="cuda")
    l_solo = [torch.zeros(3, device="cuda") for _ in range(P)]
    l_pop = [torch.zeros(3, device="cuda") for _ in range(P)]
    for rnd in range(3):
        inps = [_inputs(B, 100 * rnd + k) for k in range(P)]
        for k in range(P):
            tbl = _members([solo[k]], [inps[k]], [l_solo[k]])
            assert Lib.boatagent_sac2_update_members(tbl, 1, B, 0.9, 0.999, 1e-8, ws_solo.data_ptr(), per, None) == 0
        tbl = _members(pop, inps, l_pop)
        assert Lib.boatagent_sac2_update_members(tbl, P, B, 0.9, 0.999, 1e-8, ws.data_ptr(), ws.numel(), None) == 0
        torch.cuda.synchronize()
        for k in range(P):
            a = [p.detach() for net in solo[k].networks() for p in net.parameters()] + \
                [p.grad for p in solo[k].optimizer.params] + solo[k].optimizer.state_tensors() + [l_solo[k]]
            b = [p.detach() for net in pop[k].networks() for p in net.parameters()] + \
                [p.grad for p in pop[k].optimizer.params] + pop[k].optimizer.state_tensors() + [l_pop[k]]
            assert all(torch.equal(x, y) for x, y in zip(a, b)), f"round {rnd} member {k}"
        assert int(pop[0].optimizer.state[0]) == rnd + 1 and int(pop[-1].optimizer.state[1]) == 0
    if P > 1:
        assert not torch.equal(pop[0].temperature.log_alpha, pop[1].temperature.log_alpha)


@gpu
@pytest.mark.parametrize("learner", ["fp32", "tcgen05"])
def test_whole_loop_checkpoint_resume_is_exact(learner, tmp_path):
    """collect + learn, save, continue == fresh objects, load, continue: weights, log alpha, Adam state, ring and
    losses bit for bit.  The acting counter of the tcgen05 policy is not part of the agent's state: it is carried over
    by hand, as for SAC-v1."""
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)

    def make():
        env = S.BatchedBoatEnv(cfg, 2048, seed=3, precision="fp32", device=0, auto_reset=True)
        mem = S.ReplayBuffer(30_000, (11,), 1, precision="fp32", device=0, seed=7, as_torch=True)
        agent = ContinuousAgent(cfg, str(tmp_path), (11,), env, device=0, seed=3, memory=mem, learner_precision=learner,
                                policy_precision="tcgen05", algorithm="sac2", target_entropy=-0.5,
                                temperature_lr=1e-3)
        return env, mem, agent

    def run(env, agent, iters):
        out = []
        for _ in range(iters):
            agent.collect(env, 2)
            losses = agent.learn()
            out.append((env.obs.clone(), env.reward.clone(), torch.stack([x.detach().clone() for x in losses]),
                        agent.temperature().clone()))
        return out

    env, mem, agent = make()
    env.reset()
    run(env, agent, 10)
    torch.save({"env": env.state_dict(), "agent": agent.state_dict()}, tmp_path / "full.pt")
    acting_step = agent.tensor_core_policy().steps
    tail_a = run(env, agent, 6)
    snap_a, ring_a = _snapshot(agent), mem.state_dict()
    env2, mem2, agent2 = make()
    ck = torch.load(tmp_path / "full.pt", weights_only=False)
    env2.load_state_dict(ck["env"])
    agent2.load_state_dict(ck["agent"])
    agent2.tensor_core_policy().steps = acting_step
    tail_b = run(env2, agent2, 6)
    for x, y in zip(tail_a, tail_b):
        assert all(torch.equal(p, q) for p, q in zip(x, y))
    assert all(torch.equal(p, q) for p, q in zip(snap_a, _snapshot(agent2)))
    ring_b = mem2.state_dict()
    for k, v in ring_a.items():
        assert (torch.equal(v, ring_b[k]) if isinstance(v, torch.Tensor) else v == ring_b[k]), k
    assert "log_alpha" in ck["agent"]["networks"] and float(agent.temperature()) != 1.0
    for x in (env, env2, mem, mem2):
        x.close()


@gpu
def test_train_sac_sac2_end_to_end_and_evaluate(tmp_path, capsys):
    import evaluate_sac
    import train_sac
    base = ["--envs", "1024", "--iters", "6", "--warmup-iters", "2", "--log-every", "2", "--experiment", "6",
            "--buffer", "100000", "--policy-precision", "tcgen05", "--collect-steps", "4", "--updates-per-iter", "2",
            "--set", "agent__batch_size=256", "--algorithm", "sac2"]
    runs = {"fp32": ["--learner-precision", "fp32", "--temperature-lr", "1e-3"],
            "tcgen05": ["--learner-precision", "tcgen05", "--target-entropy", "-0.5", "--init-temperature", "0.5"],
            "population": ["--learner-precision", "tcgen05", "--population", "3"]}
    dirs = []
    for name, flags in runs.items():
        root = tmp_path / name
        summary = train_sac.main(base + flags + ["--experiments-root", str(root)])
        line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
        assert line["algorithm"] == "sac2" and summary["algorithm"] == "sac2"
        temps = line["temperature"] if name == "population" else [line["temperature"]]
        assert len(temps) == (3 if name == "population" else 1) and all(math.isfinite(t) and t > 0 for t in temps)
        assert all(math.isfinite(x) for x in (line["losses_v_pi_q"][0] if name == "population"
                                              else line["losses_v_pi_q"]))
        dirs.append(line["experiment_dirs"][0] if name == "population" else line["experiment_dir"])
    # a directory whose checkpoints a SAC-v2 agent wrote, and every run directory that saved an improving interval
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
    env = S.BatchedBoatEnv(cfg, 128, seed=0, precision="fp32", device=0, auto_reset=True)
    saved = str(tmp_path / "saved")
    a = ContinuousAgent(cfg, saved, (11,), env, device=0, memory=S.ReplayBuffer(
        1024, (11,), 1, precision="fp32", device=0, as_torch=True), algorithm="sac2")
    a.save_models()
    a.memory.close()
    env.close()
    for d in [saved] + dirs:
        ck = os.path.join(d, "checkpoints")
        if not os.path.exists(os.path.join(ck, "actor_network")):
            continue
        assert os.path.exists(os.path.join(ck, "target_critic_network_1"))
        assert os.path.exists(os.path.join(ck, "log_alpha")) and not os.path.exists(os.path.join(ck, "value_network"))
        ev = evaluate_sac.main(["--checkpoints", d, "--envs", "512", "--max-steps", "200"])
        assert ev["episodes"] + ev["running"] == 512
