"""The fused tcgen05 learner (ContinuousAgent(learner_precision="tcgen05"), csrc/learner.cu) against a PyTorch
emulation of its arithmetic, against the recorded fp32 reference update, and in the agent's workflows.

`emulate_update` is the update with bf16 rounding at exactly the points where the kernels feed the tensor cores:
fc1's inputs and weights (forward), H1 where it feeds fc2, fc2's weights, dZ2 where it feeds the input gradient
dZ2 . W2 and the weight gradient dZ2^T . H1.  Everything else is fp32.  With the rounding switched off it is the
fp32 update, which the CPU test checks against SACLearner's PyTorch restatement.
"""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import make_agent_golden as G  # noqa: E402  (test infrastructure)

import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200.continuous_agent import ContinuousAgent, SACLearner  # noqa: E402
from sac_agent_b200.networks import TensorCorePolicy  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "agent_update.npz")
TRAINED = ("actor", "critic_1", "critic_2", "value")
HEADS = {"actor": ("mean", "std"), "critic_1": ("q",), "critic_2": ("q",), "value": ("v",), "target_value": ("v",)}


def _params(nets):
    """{net: {name: fp32 tensor}} of a learner's five networks (detached copies)."""
    return {n: {k: p.detach().clone().float() for k, p in getattr(nets, n).named_parameters()} for n in G.NETS}


def _gauss_fwd(mean, raw, e, ma):
    log_std = -5.0 + 3.5 * (torch.tanh(raw) + 1.0)
    sd = torch.exp(log_std)
    u = mean + e * sd
    act = torch.tanh(u) * ma
    d = u - mean
    lp = -(d * d) / (2.0 * sd * sd) - log_std - 0.91893853320467274178 - torch.log(1.0 - act * act + 1e-6)
    return act, lp


def _gauss_bwd(mean, raw, e, ma, ga, glp):
    t = torch.tanh(raw)
    dls = 3.5 * (1.0 - t * t)
    sd = torch.exp(-5.0 + 3.5 * (t + 1.0))
    th = torch.tanh(mean + e * sd)
    act, dact = th * ma, ma * (1.0 - th * th)
    gu = ga * dact + glp * (2.0 * act * dact) / (1.0 - act * act + 1e-6)
    return gu, gu * e * sd * dls - glp * dls


def emulate_update(P, state, action, reward, new_state, done, eps, gamma, scale, max_action=1.0, rounding=True):
    """One update of the fused learner on parameters P ({net: {name: tensor}}).  Returns (grads {net: {name: g}},
    losses [3]).  state [B, 11], action [B] or [B, 1], reward [B], done [B] bool, eps [2, B] or [2, B, 1]."""
    r = (lambda t: t.to(torch.bfloat16).float()) if rounding else (lambda t: t)  # noqa: E731
    B = state.shape[0]
    a_b, e = action.reshape(B), eps.reshape(2, B)

    def fwd(n, x):
        p = P[n]
        h1 = torch.relu(r(x) @ r(p["fc1.weight"]).T + p["fc1.bias"])
        h1b = r(h1)
        h2 = torch.relu(h1b @ r(p["fc2.weight"]).T + p["fc2.bias"])
        ys = [h2 @ p[h + ".weight"][0] + p[h + ".bias"][0] for h in HEADS[n]]
        return dict(x=x, h1=h1, h1b=h1b, h2=h2, y=ys)

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

    v_ = fwd("target_value", new_state)["y"][0]
    q_hat = scale * reward + gamma * torch.where(done, torch.zeros_like(v_), v_)
    fa = fwd("actor", state)
    mean, raw = fa["y"]
    a1, lp1 = _gauss_fwd(mean, raw, e[0], max_action)
    a2, lp2 = _gauss_fwd(mean, raw, e[1], max_action)
    grads, q_a1, q_a2, dq_a2, q_sa = {}, [], [], [], []
    for n in ("critic_1", "critic_2"):
        q_a1.append(fwd(n, torch.cat([state, a1[:, None]], 1))["y"][0])
        f2 = fwd(n, torch.cat([state, a2[:, None]], 1))
        q_a2.append(f2["y"][0])
        dq_a2.append(bwd(n, f2, [torch.ones_like(a2)])[1][:, -1])
        fs = fwd(n, torch.cat([state, a_b[:, None]], 1))
        q_sa.append(fs["y"][0])
        grads[n] = bwd(n, fs, [(fs["y"][0] - q_hat) / B])[0]
    fv = fwd("value", state)
    vt = torch.minimum(q_a1[0], q_a1[1]) - lp1
    grads["value"] = bwd("value", fv, [(fv["y"][0] - vt) / B])[0]

    def share(x, y):
        return torch.where(x < y, 1.0, torch.where(x == y, 0.5, 0.0))
    ga = -(share(q_a2[0], q_a2[1]) * dq_a2[0] + share(q_a2[1], q_a2[0]) * dq_a2[1]) / B
    gm, gr = _gauss_bwd(mean, raw, e[1], max_action, ga, torch.full_like(ga, 1.0 / B))
    grads["actor"] = bwd("actor", fa, [gm, gr])[0]
    losses = torch.stack([0.5 * ((fv["y"][0] - vt) ** 2).mean(), (lp2 - torch.minimum(q_a2[0], q_a2[1])).mean(),
                          0.5 * ((q_sa[0] - q_hat) ** 2).mean() + 0.5 * ((q_sa[1] - q_hat) ** 2).mean()])
    return grads, losses


def test_emulation_without_rounding_is_the_reference_update():
    """CPU: emulate_update(rounding=False) gives SACLearner(torch_reference_math=True)'s gradients on the golden batch
    to fp32 rounding, so the emulation is the same update rule."""
    rec = np.load(GOLDEN)
    seed, batch = int(rec["meta/seed"]), int(rec["meta/batch"])
    L = SACLearner((11,), 1, np.array([1.0], dtype=np.float32), 5e-3, 3e-4, float(rec["meta/gamma"]),
                   float(rec["meta/tvn_parameter_modulation_tau"]), float(rec["meta/reward_scale"]), device="cpu",
                   torch_reference_math=True)
    w0 = G.init_weights(seed)
    for n in G.NETS:
        getattr(L, n).load_state_dict({k: torch.from_numpy(v.copy()) for k, v in w0[n].items()})
    b, noise = G.make_batch(seed, batch), G.make_noise(seed, 1, batch)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in b.items()}
    eps = torch.from_numpy(noise[0])
    P = _params(L)
    grads, losses = emulate_update(P, t["state"], t["action"], t["reward"], t["new_state"], t["done"], eps,
                                   L.gamma, L.scale, rounding=False)
    ref_losses = L.update(t["state"], t["action"], t["reward"], t["new_state"], t["done"], eps_sample=eps[0],
                          eps_rsample=eps[1])
    for n in TRAINED:
        for k, p in getattr(L, n).named_parameters():
            g, ref = grads[n][k], p.grad
            assert (g - ref).abs().max().item() <= 2e-5 * ref.abs().max().item() + 1e-9, (n, k)
    assert torch.allclose(losses, torch.stack(list(ref_losses)), rtol=1e-5, atol=1e-7)


# ----------------------------------------------------------------------------------------------------------------
def _env_stub():
    return type("E", (), {"action_space": S.Box(low=-1, high=1, dtype=np.float32)})()


def _agent(batch, learner_precision="tcgen05", seed=0, **kw):
    cfg = S.load_config(agent__batch_size=batch)
    mem = kw.pop("memory", None) or S.ReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    torch.manual_seed(seed)
    return ContinuousAgent(cfg, None, (11,), _env_stub(), device=0, memory=mem, learner_precision=learner_precision,
                           **kw)


def _random_batch(B, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    st = torch.rand(B, 11, generator=g) * 2 - 1
    return dict(state=st.cuda(), action=(torch.rand(B, 1, generator=g) * 2 - 1).cuda(),
                reward=torch.randn(B, generator=g).cuda(), new_state=(st + 0.1 * torch.randn(B, 11, generator=g)).cuda(),
                done=(torch.rand(B, generator=g) < 0.1).cuda(), eps=torch.randn(2, B, 1, generator=g).cuda())


def _adam_emulation(agent, P, grads):
    """What the kernels' Adam + Polyak step makes of the parameters P with gradients `grads` (fp32, DeviceAdam order)."""
    o = agent.learner.optimizer
    t = int(o.state[0]) + 1
    b1, b2 = o.betas
    bc1, bc2s = 1.0 - b1 ** t, (1.0 - b2 ** t) ** 0.5
    names = [(n, k) for n in TRAINED for k, _ in getattr(agent.learner, n).named_parameters()]
    order = {nk: i for i, nk in enumerate(names)}
    new = {n: dict(P[n]) for n in G.NETS}
    for (n, k), i in order.items():
        g, m, v = grads[n][k], o.exp_avg[i].float(), o.exp_avg_sq[i].float()
        m2 = m + (g - m) * (1 - b1)
        v2 = v * b2 + (1 - b2) * g * g
        new[n][k] = P[n][k] - (o._slots[i].lr / bc1) * (m2 / (v2.sqrt() / bc2s + o.eps))
        if n == "value":
            new["target_value"][k] = o.tau * new[n][k] + (1 - o.tau) * P["target_value"][k]
    return new


def _check_update(agent, batch, grad_tol=2e-3, loss_rtol=2e-3):
    """One learn_from on `batch`, compared with the emulation from the weights before it: every .grad within
    grad_tol of the tensor's largest gradient, the weights within the lr-based tolerance, the three losses."""
    L = agent.learner
    P = _params(L)
    grads, losses = emulate_update(P, batch["state"], batch["action"], batch["reward"], batch["new_state"],
                                   batch["done"], batch["eps"], L.gamma, L.scale)
    expect = _adam_emulation(agent, P, grads)
    got_losses = agent.learn_from(batch["state"], batch["action"], batch["reward"], batch["new_state"],
                                  batch["done"].to(torch.uint8), eps=batch["eps"])
    torch.cuda.synchronize()
    worst = {}
    for n in TRAINED:
        lr = float(L.optimizer._slots[0 if n == "actor" else 8].lr)
        for k, p in getattr(L, n).named_parameters():
            ref = grads[n][k]
            err = (p.grad - ref).abs().max().item() / max(ref.abs().max().item(), 1e-12)
            worst[f"{n}.{k}"] = err
            assert err <= grad_tol, (n, k, err)
            werr = (p.detach() - expect[n][k]).abs()
            assert (werr > 1e-6 + 0.02 * lr).float().mean().item() <= 0.002, (n, k, werr.max().item())
    for k, p in L.target_value.named_parameters():
        assert (p.detach() - expect["target_value"][k]).abs().max().item() <= 1e-6 + 0.02 * 3e-4 * 0.005 + 1e-7
    got = torch.stack([x.detach() for x in got_losses])
    assert torch.allclose(got, losses, rtol=loss_rtol, atol=1e-6), (got, losses)
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_fused_update_matches_emulation(B):
    agent = _agent(B, seed=B)
    with torch.no_grad():   # weights away from the initialisation's symmetric regime
        for p in agent.learner._actor_params + agent.learner._critic_params + agent.learner._value_params:
            p.add_(0.02 * torch.randn_like(p))
        agent.learner.update_network_parameters(tau=1.0)
    for u in range(3):
        worst = _check_update(agent, _random_batch(B, 100 * B + u))
    print(f"B={B}: worst |grad - emulation| / max|grad| = {max(worst.values()):.2e} ({max(worst, key=worst.get)})")
    assert int(agent.learner.optimizer.state[0]) == 3 and int(agent.learner.optimizer.state[1]) == 0
    agent.memory.close()


# bf16 margins measured on the golden batch (B = 1024) against the recorded fp32 run of the reference's own learn(),
# updates 1 and 3.  Gradients: the worst sampled |ours - ref| over the tensor's largest |ref|.  Weights: the first Adam
# steps move every weight by ~lr * sign(g), so where bf16 flips the sign of a near-zero gradient the weight lands
# ~2 lr away; the test bounds the share of sampled weights more than lr / 2 away.  A wrong sign or a missing term of
# a network's gradient moves most of that network's weights by ~lr to 2 lr and its gradients by O(1) of their maximum.
# Measured on an NVIDIA B200 (the update is bit-reproducible, so every run gives these): gradients 1.98e-2
# (u3/actor/fc1.weight), weights 0.98 % of the sampled positions (u3/value/fc1.weight).  The bounds leave 1.5x / 2x.
GOLDEN_GRAD_TOL, GOLDEN_W_FRAC = 0.03, 0.02


@pytest.mark.gpu
def test_fused_update_against_recorded_reference():
    rec = np.load(GOLDEN)
    seed, n_updates, batch = int(rec["meta/seed"]), int(rec["meta/n_updates"]), int(rec["meta/batch"])
    b, noise = G.make_batch(seed, batch), G.make_noise(seed, n_updates, batch)
    agent = _agent(batch)
    L = agent.learner
    w0 = G.init_weights(seed)
    for n in G.NETS:
        getattr(L, n).load_state_dict({k: torch.from_numpy(v.copy()) for k, v in w0[n].items()})
    lr_of = {n: float(rec["meta/learning_rate_alpha"] if n == "actor" else rec["meta/learning_rate_beta"]) for n in G.NETS}
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in b.items()}
    errs = {}
    for u in range(1, n_updates + 1):
        agent.learn_from(t["state"], t["action"], t["reward"], t["new_state"], t["done"].to(torch.uint8),
                         eps=torch.from_numpy(noise[u - 1]))
        if u not in rec["meta/record_after"]:
            continue
        for n in G.NETS:
            for k, p in getattr(L, n).named_parameters():
                for kind in ("w", "g"):
                    key = f"u{u}/{n}/{k}/{kind}"
                    if key + "@" not in rec:
                        continue
                    tt = p if kind == "w" else p.grad
                    ours = tt.detach().float().cpu().numpy().reshape(-1)[G.sample_positions(tuple(p.shape), key)]
                    ref = rec[key + "@"]
                    d = np.abs(ours - ref)
                    errs[key] = (float(d.max() / max(np.abs(ref).max(), 1e-12)) if kind == "g"
                                 else float(np.mean(d > 0.5 * lr_of[n])))
    g_worst = max((v, k) for k, v in errs.items() if k.endswith("/g"))
    w_worst = max((v, k) for k, v in errs.items() if k.endswith("/w"))
    print(f"golden: worst grad error {g_worst[0]:.3e} of max|g| ({g_worst[1]}), "
          f"worst share of weights > lr/2 away {w_worst[0]:.3e} ({w_worst[1]})")
    assert g_worst[0] <= GOLDEN_GRAD_TOL and w_worst[0] <= GOLDEN_W_FRAC, (g_worst, w_worst)
    agent.memory.close()


def _snapshot(agent):
    L, o = agent.learner, agent.learner.optimizer
    out = [p.detach().clone() for net in L.networks() for p in net.parameters()]
    out += [p.grad.clone() for p in o.params] + [t.clone() for t in o.state_tensors()]
    return out


@pytest.mark.gpu
def test_fused_update_is_bit_reproducible():
    agents = [_agent(1024, seed=4) for _ in range(2)]
    agents[1].load_state_dict(agents[0].state_dict())
    for u in range(3):
        b = _random_batch(1024, u)
        ls = [a.learn_from(b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8), eps=b["eps"])
              for a in agents]
        assert all(torch.equal(x, y) for x, y in zip(ls[0], ls[1]))
    s0, s1 = _snapshot(agents[0]), _snapshot(agents[1])
    assert all(torch.equal(x, y) for x, y in zip(s0, s1))
    for a in agents:
        a.memory.close()


@pytest.mark.gpu
def test_whole_sac_loop_checkpoint_resume_is_exact_with_fused_learner(tmp_path):
    """test_agent_golden's resume scenario with learner_precision="tcgen05": save -> keep running == fresh objects ->
    load -> run, bit for bit."""
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)

    def make():
        env = S.BatchedBoatEnv(cfg, 2048, seed=3, precision="fp32", device=0, auto_reset=True)
        mem = S.ReplayBuffer(30_000, (11,), 1, precision="fp32", device=0, seed=7, as_torch=True)
        agent = ContinuousAgent(cfg, str(tmp_path), (11,), env, device=0, seed=3, memory=mem, learner_precision="tcgen05")
        return env, mem, agent

    def run(env, agent, iters):
        out = []
        for _ in range(iters):
            a = agent.choose_action(env.obs)
            agent.step_and_remember(env, a.squeeze(-1))
            losses = agent.learn()
            out.append((env.obs.clone(), env.reward.clone(), torch.stack([x.detach().clone() for x in losses])))
        return out

    os.makedirs(tmp_path / "checkpoints", exist_ok=True)
    env, mem, agent = make()
    env.reset()
    run(env, agent, 25)
    torch.save({"env": env.state_dict(), "agent": agent.state_dict()}, tmp_path / "full.pt")
    tail_a = run(env, agent, 12)
    weights_a = _snapshot(agent)
    env2, mem2, agent2 = make()
    ck = torch.load(tmp_path / "full.pt", weights_only=False)
    env2.load_state_dict(ck["env"])
    agent2.load_state_dict(ck["agent"])
    tail_b = run(env2, agent2, 12)
    for (o1, r1, l1), (o2, r2, l2) in zip(tail_a, tail_b):
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(l1, l2)
    assert all(torch.equal(p, q) for p, q in zip(weights_a, _snapshot(agent2)))
    for x in (env, env2, mem, mem2):
        x.close()


@pytest.mark.gpu
def test_training_state_moves_between_learners(tmp_path):
    """A training state saved under one learner loads into the other and training continues from it: the loaded
    agent's next update is the emulation's update of the loaded weights and Adam state."""
    for src, dst in (("fp32", "tcgen05"), ("tcgen05", "fp32")):
        a = _agent(256, learner_precision=src, seed=1)
        for u in range(2):
            b = _random_batch(256, u)
            a.learn_from(b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8), eps=b["eps"])
        path = a.save_training_state(str(tmp_path / f"{src}.pt"))
        c = _agent(256, learner_precision=dst, seed=2)
        c.load_training_state(path)
        assert c.updates == 2 and int(c.learner.optimizer.state[0]) == 2
        weights = lambda x: [p for net in x.learner.networks() for p in net.parameters()]  # noqa: E731
        assert all(torch.equal(p, q) for p, q in zip(weights(a), weights(c)))
        assert all(torch.equal(p, q) for p, q in zip(a.learner.optimizer.state_tensors(),
                                                     c.learner.optimizer.state_tensors()))
        if dst == "tcgen05":
            _check_update(c, _random_batch(256, 9))
        else:
            b = _random_batch(256, 9)
            ls = c.learn_from(b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8), eps=b["eps"])
            assert all(torch.isfinite(x).item() for x in ls) and int(c.learner.optimizer.state[0]) == 3
        a.memory.close(); c.memory.close()


@pytest.mark.gpu
def test_changed_hyperparameters_reach_the_next_update():
    agent = _agent(512, seed=3)
    b = _random_batch(512, 1)
    agent.learn_from(b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8), eps=b["eps"])
    agent.set_hyperparameters(alpha=1e-3, beta=7e-4, gamma=0.9, tau=0.05)
    assert agent.hyperparameters() == pytest.approx({"alpha": 1e-3, "beta": 7e-4, "gamma": 0.9, "tau": 0.05})
    _check_update(agent, _random_batch(512, 2))
    agent.memory.close()


@pytest.mark.gpu
def test_fused_learner_in_the_training_loops():
    """OverlappedActorLearner, collect + learn and the tcgen05 policy's refresh with the fused learner."""
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=512)
    env = S.BatchedBoatEnv(cfg, 8192, seed=5, precision="fp32", device=0, auto_reset=True)
    mem = S.ReplayBuffer(100_000, (11,), 1, precision="fp32", device=0, as_torch=True)
    agent = ContinuousAgent(cfg, None, (11,), env, device=0, seed=5, memory=mem, learner_precision="tcgen05",
                            policy_precision="tcgen05")
    env.reset()
    pipe = S.OverlappedActorLearner(agent, env)
    for _ in range(10):
        losses = pipe.step()
    pipe.finish()
    torch.cuda.synchronize()
    assert agent.updates == 10 and all(torch.isfinite(x).item() for x in losses)
    assert all(torch.equal(p, q) for p, q in zip(pipe.acting[1].parameters(), agent.actor.parameters()))
    for _ in range(3):
        agent.collect(env, 4)
        losses = agent.learn()
    torch.cuda.synchronize()
    assert agent.updates == 13 and all(torch.isfinite(x).item() for x in losses)
    pol = agent.tensor_core_policy()
    obs, eps = env.obs.clone(), torch.randn(8192, 1, device="cuda")
    fresh = TensorCorePolicy(agent.actor).act(obs, eps)
    assert torch.equal(pol.act(obs, eps), fresh)     # learn() refreshed the packed copy
    env.close(); mem.close()


@pytest.mark.gpu
def test_fused_learner_errors():
    from sac_agent_b200 import _lib
    cfg = S.load_config(agent__batch_size=256)
    mem = S.ReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    with pytest.raises(ValueError):
        ContinuousAgent(cfg, None, (11,), _env_stub(), device=0, memory=mem, learner_precision="bf16")
    for bad in (100, 200, 64):
        with pytest.raises(ValueError):
            ContinuousAgent(S.load_config(agent__batch_size=bad), None, (11,), _env_stub(), device=0, memory=mem,
                            learner_precision="tcgen05")
    with pytest.raises(ValueError):
        ContinuousAgent(cfg, None, (12,), _env_stub(), device=0, memory=mem, learner_precision="tcgen05")
    two = type("E", (), {"action_space": S.Box(low=-np.ones(2), high=np.ones(2), dtype=np.float32)})()
    with pytest.raises(ValueError):
        ContinuousAgent(cfg, None, (11,), two, device=0, memory=mem, learner_precision="tcgen05")

    L = _lib.lib()
    EINVAL, EALIGN = -1, -7
    assert L.boatagent_sac_update_workspace_bytes(0) == EINVAL and L.boatagent_sac_update_workspace_bytes(130) == EINVAL
    agent = ContinuousAgent(cfg, None, (11,), _env_stub(), device=0, memory=mem, learner_precision="tcgen05")
    o = agent.learner.optimizer
    for k, p in enumerate(o.params):
        p.grad = torch.zeros_like(p)
        o._slots[k].grad = p.grad.data_ptr()
    s, a, r, s2, d = agent._batch
    x = agent._eps

    def call(**kw):
        args = dict(state=s.data_ptr(), action=a.data_ptr(), reward=r.data_ptr(), new_state=s2.data_ptr(),
                    done=d.data_ptr(), eps=x.data_ptr(), max_action=agent.actor.max_action.data_ptr(), batch=256,
                    slots=o._slots, n_slots=26, state_ptr=o.state.data_ptr(), losses=agent._loss_buf.data_ptr(),
                    ws=agent._ws.data_ptr(), ws_bytes=agent._ws.numel())
        args.update(kw)
        return L.boatagent_sac_update(args["state"], args["action"], args["reward"], args["new_state"], args["done"],
                                      args["eps"], args["max_action"], args["batch"], 0.99, 10.0, args["slots"],
                                      args["n_slots"], 0.9, 0.999, 1e-8, 0.005, args["state_ptr"], args["losses"],
                                      args["ws"], args["ws_bytes"], None)

    for name in ("state", "action", "reward", "new_state", "done", "eps", "max_action", "slots", "state_ptr", "losses",
                 "ws"):
        assert call(**{name: None}) == EINVAL, name
    for bad in (0, 100, 384):   # 384: a valid batch, but larger than the workspace
        assert call(batch=bad) == EINVAL, bad
    assert call(n_slots=25) == EINVAL
    assert call(ws_bytes=agent._ws.numel() - 1) == EINVAL
    assert call(ws=agent._ws.data_ptr() + 4) == EALIGN
    keep = o._slots[2].numel
    o._slots[2].numel = keep - 1
    assert call() == EINVAL
    o._slots[2].numel = keep
    keep = o._slots[20].target
    o._slots[20].target = None
    assert call() == EINVAL
    o._slots[20].target = keep
    o._slots[0].target = o._slots[0].param
    assert call() == EINVAL
    o._slots[0].target = None
    keep = o._slots[5].grad
    o._slots[5].grad = None
    assert call() == EINVAL
    o._slots[5].grad = keep
    torch.cuda.synchronize()
    assert int(o.state[0]) == 0   # nothing ran
    assert call() == 0
    torch.cuda.synchronize()
    assert int(o.state[0]) == 1
    mem.close()
