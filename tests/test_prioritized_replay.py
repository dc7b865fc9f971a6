"""Prioritized experience replay (PrioritizedReplayBuffer, boatper_*, the prioritized fused learner updates,
ContinuousAgent(prioritized=True), train_sac --prioritized).

A numpy restatement of the device sum tree (RefTree: the same 1024 fan-out, the same fixed-order fp64 block sums, the
same stratified descent with its clamp, the same weights and max-of-duplicates update) is checked against a brute-force
cumulative-sum sampler on the CPU, and the device tree against it exactly on the GPU.  The weighted learners are held
to a float64 restatement (CPU), to the unweighted learners when every weight is 1, and the fused kernels to a weighted
bf16 emulation (GPU).
"""
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
from sac_agent_b200.continuous_agent import ContinuousAgent, SAC2Learner, SACLearner  # noqa: E402
from boat_testlib import philox4x32_10, set_mem_cntr  # noqa: E402
from test_gpu_learner import _env_stub, _gauss_fwd, emulate_update  # noqa: E402
from test_sac2 import emulate_update_sac2  # noqa: E402

gpu = pytest.mark.gpu
FAN = 1024
EINVAL = -1


# ---- the numpy restatement of the device tree (csrc/priority.cu) ----------------------------------------------------

def _chunk_sums(blocks):
    """[n, 1024] -> [n, 32]: lane l's entries 32 l .. 32 l + 31 summed in order in fp64 (chunk_sum)."""
    x = blocks.reshape(-1, 32, 32).astype(np.float64)
    s = np.zeros(x.shape[:2])
    for i in range(32):
        s = s + x[:, :, i]
    return s


def _scan(v):
    """Inclusive prefix sums over the last axis of 32, lane l adding lane l - o for o = 1, 2, 4, 8, 16 (warp_scan)."""
    v = v.copy()
    for o in (1, 2, 4, 8, 16):
        u = v.copy()
        v[..., o:] = u[..., o:] + u[..., :-o]
    return v


def _pick(t, incl, own):
    """First lane with a non-zero share whose prefix exceeds t, else the last lane with a non-zero share, else 0
    (pick_lane)."""
    nz = own > 0
    hit = (t[:, None] < incl) & nz
    last = 31 - np.argmax(nz[:, ::-1], axis=1)
    return np.where(hit.any(1), np.argmax(hit, axis=1), np.where(nz.any(1), last, 0))


def _descend(arr, b, t):
    """One block per row (b: block indices, t: targets) -> (entry within the block, residual t) (descend)."""
    rows = np.arange(len(b))
    blk = arr[(b[:, None] * FAN + np.arange(FAN)[None, :])].astype(np.float64)
    c = _chunk_sums(blk)
    S_ = _scan(c)
    L = _pick(t, S_, c)
    t = t - np.where(L > 0, S_[rows, np.maximum(L - 1, 0)], 0.0)
    v = blk.reshape(-1, 32, 32)[rows, L]
    V = _scan(v)
    I_ = _pick(t, V, v)
    t = t - np.where(I_ > 0, V[rows, np.maximum(I_ - 1, 0)], 0.0)
    return 32 * L + I_, t


class RefTree:
    def __init__(self, mem_size):
        self.mem_size = mem_size
        self.count = [mem_size]
        while True:
            self.count.append(-(-self.count[-1] // FAN))
            if self.count[-1] == 1:
                break
        pad = lambda n: -(-n // FAN) * FAN  # noqa: E731
        self.levels = [np.zeros(pad(mem_size), np.float32)] + [np.zeros(pad(n), np.float64) for n in self.count[1:]]
        self.max_p = np.float32(1.0)
        self.filled = 0

    def resum(self):   # every block sum is a function of its children: a full resum equals the device's partial one
        for k in range(1, len(self.levels)):
            child = self.levels[k - 1][:self.count[k] * FAN]
            self.levels[k][:self.count[k]] = _scan(_chunk_sums(child.reshape(-1, FAN)))[:, 31]

    def fill(self, first, n):
        if n > self.mem_size:
            first, n = first + n - self.mem_size, self.mem_size
        self.levels[0][(first + np.arange(n)) % self.mem_size] = self.max_p
        self.filled = min(self.mem_size, max(self.filled, first + n))
        self.resum()

    def targets(self, batch, seed, counter):
        j = np.arange(batch, dtype=np.uint64)
        c = int(counter)
        r = philox4x32_10(j, j >> np.uint64(32), c, 0xE0000000 | ((c >> 32) & 0x0FFFFFFF), int(seed), int(seed) >> 32)
        u = ((r[0] >> np.uint64(5)) * np.uint64(67108864) + (r[1] >> np.uint64(6))).astype(np.float64) * 2.0 ** -53
        return ((j.astype(np.float64) + u) / batch) * self.levels[-1][0]

    def descend(self, t):
        b = np.zeros(len(t), np.int64)
        for k in range(len(self.levels) - 2, 0, -1):
            e, t = _descend(self.levels[k], b, t)
            b = b * FAN + e
        e, _ = _descend(self.levels[0], b, t)
        return b * FAN + e

    def sample(self, batch, seed, counter, beta):
        idx = self.descend(self.targets(batch, seed, counter))
        p = self.levels[0][idx].astype(np.float64)
        return idx, np.power(p.min() / p, beta).astype(np.float32)

    def update(self, idx, td, alpha, eps):
        p = np.power((td.astype(np.float32) + np.float32(eps)).astype(np.float64), alpha).astype(np.float32)
        self.levels[0][idx] = 0
        np.maximum.at(self.levels[0], idx, p)
        self.max_p = max(self.max_p, p.max())
        self.resum()


def _brute(leaves, t):
    """The slot of each target by a cumulative sum over every leaf."""
    return np.searchsorted(np.cumsum(leaves.astype(np.float64)), t, side="right")


@pytest.mark.parametrize("case", ["equal", "one_hot", "zero_tail", "wrapped", "skewed"])
def test_reference_tree_matches_brute_force_sampler(case):
    """Integer priorities keep every sum exact, so the stratified descent must land where a cumulative sum does."""
    rng = np.random.default_rng(7)
    n = 5000
    T = RefTree(n)
    if case == "equal":
        T.fill(0, n)
    elif case == "one_hot":
        T.fill(0, 1)
        T.levels[0][0] = 0
        T.levels[0][3071] = 5
        T.resum()
    elif case == "zero_tail":
        T.fill(0, 2100)
    elif case == "wrapped":
        T.fill(0, n)
        T.fill(n - 300, 700)   # rows n - 300 .. n + 399: slots n - 300 .. n - 1 and 0 .. 399
        T.levels[0][:] = 0
        T.levels[0][np.r_[n - 300:n, 0:400]] = 2
        T.resum()
    else:
        T.fill(0, n)
        T.levels[0][:n] = rng.integers(1, 1000, n) ** 2 % 977
        T.resum()
    leaves = T.levels[0][:n]
    assert T.levels[-1][0] == leaves.astype(np.float64).sum()
    t = T.targets(4096, 3, 11)
    got = T.descend(t)
    assert np.array_equal(got, _brute(leaves, t))
    assert (leaves[got] > 0).all()


def test_reference_tree_clamps_rounding_past_the_last_nonzero_leaf():
    """A target on or past the total (fp rounding at the last stratum) returns the last non-zero leaf, never a zero
    leaf beyond the filled ones; so does a target past a block's own sum."""
    T = RefTree(3000)
    T.fill(0, 2100)
    T.levels[0][:2100] = np.random.default_rng(1).random(2100).astype(np.float32) + 0.1
    T.resum()
    total = T.levels[-1][0]
    for t in (total, np.nextafter(total, np.inf), total * (1 + 1e-12)):
        assert T.descend(np.array([t]))[0] == 2099
    # past block 0's sum but within rounding of it: the last non-zero leaf of block 0 (1023)
    e, _ = _descend(T.levels[0], np.array([0]), np.array([T.levels[1][0] * (1 + 1e-15)]))
    assert e[0] == 1023


def test_reference_weights_and_duplicate_update():
    T = RefTree(2048)
    T.fill(0, 2048)
    idx = np.array([5, 9, 5, 2047, 9, 5])
    td = np.array([1.0, 0.5, 3.0, 0.25, 0.1, 2.0], np.float32)
    T.update(idx, td, 0.7, 1e-3)
    p = lambda x: np.float32(np.power(np.float64(np.float32(x) + np.float32(1e-3)), 0.7))  # noqa: E731
    assert T.levels[0][5] == p(3.0) and T.levels[0][9] == p(0.5) and T.levels[0][2047] == p(0.25)
    assert T.max_p == p(3.0)
    idx, w = T.sample(512, 0, 0, 0.5)
    pr = T.levels[0][idx].astype(np.float64)
    ref = np.power(T.filled * pr / T.levels[-1][0], -0.5)
    assert np.allclose(w, ref / ref.max(), rtol=1e-6) and w.max() == 1.0


def test_per_stream_is_philox_in_its_own_domain():
    """The stratified draws' Philox blocks are (row lo, hi, counter lo, 0xE0000000 | counter hi), key = seed: distinct
    from the acting (0xD), replay (0xB), action (0xA) and toy (0xC) domains."""
    T = RefTree(1024)
    T.fill(0, 1024)
    seed, counter = 0x1234_5678_9ABC, (5 << 32) | 17
    r = philox4x32_10(np.uint64(3), 0, counter & 0xFFFFFFFF, 0xE0000005, seed & 0xFFFFFFFF, seed >> 32)
    u = (int(r[0]) >> 5) * 67108864 + (int(r[1]) >> 6)
    assert T.targets(8, seed, counter)[3] == ((3 + u * 2.0 ** -53) / 8) * 1024.0


# ---- the weighted fp32 learners (CPU) -------------------------------------------------------------------------------

def _cpu_batch(B, seed):
    g = torch.Generator().manual_seed(seed)
    st = torch.rand(B, 11, generator=g) * 2 - 1
    return dict(state=st, action=torch.rand(B, 1, generator=g) * 2 - 1, reward=torch.randn(B, generator=g),
                new_state=st + 0.1 * torch.randn(B, 11, generator=g), done=torch.rand(B, generator=g) < 0.2,
                eps=torch.randn(2, B, 1, generator=g))


def _learner(algo, seed):
    torch.manual_seed(seed)
    cls = SAC2Learner if algo == "sac2" else SACLearner
    L = cls((11,), 1, np.ones(1, np.float32), 5e-3, 3e-4, 0.99, 0.005, 10.0, device="cpu", torch_reference_math=True)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for net in L.networks():
            for p in net.parameters():
                p.add_(0.02 * torch.randn(p.shape, generator=g))
    return L


def _grads(L):
    params = L.optimizer_params() if hasattr(L, "optimizer_params") else \
        L._actor_params + L._critic_params + L._value_params
    return [p.grad.clone() for p in params] + [p.detach().clone() for p in params]


def _update(L, b, **kw):
    return L.update(b["state"], b["action"], b["reward"], b["new_state"], b["done"], eps_sample=b["eps"][0],
                    eps_rsample=b["eps"][1], **kw)


@pytest.mark.parametrize("algo", ["sac1", "sac2"])
def test_unit_weights_are_the_unweighted_learner_bit_for_bit(algo):
    b = _cpu_batch(256, 4)
    La, Lb = _learner(algo, 3), _learner(algo, 3)
    la = _update(La, b)
    td = torch.zeros(256)
    lb = _update(Lb, b, weights=torch.ones(256), td_out=td)
    assert all(torch.equal(x, y) for x, y in zip(la, lb))
    assert all(torch.equal(x, y) for x, y in zip(_grads(La), _grads(Lb)))
    assert (td > 0).all()


def _critic_f64(L, b, w, algo):
    """The weighted critic loss, its critic gradients and the TD errors written out in float64 with autograd."""
    s, a, r, s2 = (b[k].double() for k in ("state", "action", "reward", "new_state"))
    done = b["done"].double()

    def mlp(net, x):
        h = torch.relu(x @ net.fc1.weight.double().T + net.fc1.bias.double())
        h = torch.relu(h @ net.fc2.weight.double().T + net.fc2.bias.double())
        return h

    def q(net, x, act, W=None):
        W = W or {k: v.double() for k, v in net.named_parameters()}
        h = torch.relu(torch.cat([x, act], 1) @ W["fc1.weight"].T + W["fc1.bias"])
        h = torch.relu(h @ W["fc2.weight"].T + W["fc2.bias"])
        return (h @ W["q.weight"].T + W["q.bias"]).view(-1)
    with torch.no_grad():
        if algo == "sac1":
            v = mlp(L.target_value, s2) @ L.target_value.v.weight.double().T + L.target_value.v.bias.double()
            target = 10.0 * r + 0.99 * (1 - done) * v.view(-1)
        else:
            la = L.temperature.log_alpha.detach()
            mean, raw = [t.double() for t in L.actor.forward(b["new_state"])]
            log_std = -5.0 + 3.5 * (torch.tanh(raw) + 1.0)
            std = log_std.exp()
            u = mean + b["eps"][0].double() * std
            act = torch.tanh(u)
            lp = (-((u - mean) ** 2) / (2 * std * std) - log_std - 0.5 * math.log(2 * math.pi)
                  - torch.log(1 - act ** 2 + 1e-6)).sum(1)
            qt = torch.min(q(L.target_critic_1, s2, act), q(L.target_critic_2, s2, act))
            target = 10.0 * r + 0.99 * (1 - done) * (qt - la.double().exp() * lp)
    Ws = [{k: v.double().clone().requires_grad_(True) for k, v in net.named_parameters()}
          for net in (L.critic_1, L.critic_2)]
    q1, q2 = q(L.critic_1, s, a, Ws[0]), q(L.critic_2, s, a, Ws[1])
    w = w.double()
    loss = 0.5 * (w * (q1 - target) ** 2).mean() + 0.5 * (w * (q2 - target) ** 2).mean()
    grads = torch.autograd.grad(loss, list(Ws[0].values()) + list(Ws[1].values()))
    return loss.detach(), grads, (0.5 * ((q1 - target).abs() + (q2 - target).abs())).detach()


@pytest.mark.parametrize("algo", ["sac1", "sac2"])
def test_weighted_learner_is_the_float64_restatement(algo):
    b = _cpu_batch(256, 5)
    L = _learner(algo, 6)
    w = torch.rand(256, generator=torch.Generator().manual_seed(8)) * 0.9 + 0.1
    ref_loss, ref_g, ref_td = _critic_f64(L, b, w, algo)
    td = torch.zeros(256)
    losses = _update(L, b, weights=w, td_out=td)
    got = [p.grad for p in L._critic_params]
    for g, r in zip(got, ref_g):
        assert (g.double() - r).abs().max().item() <= 1e-5 * r.abs().max().item() + 1e-12
    assert abs(losses[2].item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    assert torch.allclose(td.double(), ref_td, rtol=1e-5, atol=1e-5)


# ---- rejections (CPU) ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("flags", [
    ["--priority-alpha", "0.5"], ["--priority-beta", "0.5"], ["--priority-beta-updates", "10"], ["--priority-eps", "0.1"],
    ["--prioritized", "--data-parallel"], ["--prioritized", "--population", "2"], ["--prioritized", "--overlap"],
    ["--prioritized", "--priority-alpha", "-1"], ["--prioritized", "--priority-beta", "1.5"],
    ["--prioritized", "--priority-eps", "0"]])
def test_train_sac_rejects_priority_combinations_before_cuda_work(flags, monkeypatch):
    import train_sac
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("CUDA work before the argument checks"))
    with pytest.raises(SystemExit):
        train_sac.main(flags)


def test_train_sac_rejects_prioritized_rounds_across_ranks(monkeypatch):
    import train_sac
    monkeypatch.setattr(S.sharding, "dist_info", lambda: (0, 0, 2))
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("CUDA work before the argument checks"))
    with pytest.raises(SystemExit):
        train_sac.main(["--prioritized", "--pbt-every", "5"])


@pytest.mark.parametrize("kw", [dict(priority_alpha=0.5), dict(priority_beta_updates=3),
                                dict(prioritized=True, data_parallel=True),
                                dict(prioritized=True, priority_eps=0.0), dict(prioritized=True, priority_beta=-0.1),
                                dict(prioritized=True, memory="uniform")])
def test_agent_rejects_priority_combinations_before_cuda_work(kw, monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: pytest.fail("CUDA work before the argument checks"))
    if kw.get("memory") == "uniform":
        kw["memory"] = object.__new__(S.ReplayBuffer)
    with pytest.raises(ValueError):
        ContinuousAgent(S.load_config(), None, (11,), _env_stub(), **kw)


def test_overlapped_pipeline_rejects_a_prioritized_agent():
    agent = type("A", (), {"data_parallel": False, "prioritized": True})()
    with pytest.raises(ValueError, match="prioritized"):
        S.OverlappedActorLearner(agent, None)


# ---- GPU: the device tree --------------------------------------------------------------------------------------------

def _tree_equal(mem, T):
    n = mem.tree_levels()
    assert n == len(T.levels)
    for k in range(n):
        got = mem.tree_level(k).cpu().numpy()
        assert np.array_equal(got, T.levels[k][:T.count[k]]), k
    assert mem.tree_level(-1).item() == T.max_p


@gpu
@pytest.mark.parametrize("log2", [20, 25])
def test_device_tree_fills_updates_and_draws_as_the_reference(log2):
    n = 1 << log2
    mem = S.PrioritizedReplayBuffer(n, (11,), 1, precision="fp32", device=0, seed=9, as_torch=True, alpha=0.6,
                                    eps=1e-3)
    T = RefTree(n)
    rng = np.random.default_rng(log2)
    row = 0
    for step, rows in enumerate((n // 3, n // 2, n // 4 + 12345)):   # the third fill wraps the ring
        set_mem_cntr(mem, row + rows)
        T.fill(row, rows)
        row += rows
        for batch in (128, 1024, 4096):
            s, a, r, s2, d, idx, w = mem.sample_buffer(batch, beta=0.4 + 0.2 * step)
            ridx, rw = T.sample(batch, 9, mem._per_samples - 1, 0.4 + 0.2 * step)
            assert np.array_equal(idx.cpu().numpy(), ridx), (step, batch)
            assert np.array_equal(w.cpu().numpy(), rw), (step, batch)
            td = torch.from_numpy(rng.exponential(2.0, batch).astype(np.float32))
            dup = idx.clone()
            dup[batch // 2:batch // 2 + 64] = dup[:64]   # slots drawn twice in one update
            mem.update_priorities(dup, td.cuda())
            T.update(dup.cpu().numpy(), td.numpy(), 0.6, 1e-3)
        mem.check()
        _tree_equal(mem, T)
    mem.close()


@gpu
def test_update_flags_indices_outside_the_ring():
    mem = S.PrioritizedReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    set_mem_cntr(mem, 4096)
    mem.sample_buffer(128)
    before = mem.tree_level(0).clone()
    mem.update_priorities(torch.tensor([5, 4096, -1], device="cuda"), torch.tensor([1.0, 2.0, 3.0], device="cuda"))
    with pytest.raises(S.BoatEnvError):
        mem.check()
    mem.check()   # the flag is cleared
    after = mem.tree_level(0)
    assert after[5] != before[5] and torch.equal(after[6:], before[6:])
    # a negative TD error is rejected even where the exponent would make its priority positive
    sq = S.PrioritizedReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True, alpha=2.0)
    set_mem_cntr(sq, 4096)
    sq.sample_buffer(128)
    sq.update_priorities(torch.tensor([7, 8], device="cuda"), torch.tensor([-3.0, float("nan")], device="cuda"))
    with pytest.raises(S.BoatEnvError):
        sq.check()
    assert sq.tree_level(0)[7].item() == 1.0 and sq.tree_level(0)[8].item() == 1.0
    sq.close()
    L, h = mem._L, mem._p
    z = torch.zeros(4, dtype=torch.int64, device="cuda")
    f = torch.zeros(4, device="cuda")
    st = mem._stream()
    assert L.boatper_sample(h, 0, 0, 0, 0.4, z.data_ptr(), f.data_ptr(), st) == EINVAL
    assert L.boatper_sample(h, 4, 0, 0, -0.1, z.data_ptr(), f.data_ptr(), st) == EINVAL
    assert L.boatper_sample(h, 4, 0, 0, 0.4, None, f.data_ptr(), st) == EINVAL
    assert L.boatper_update(h, 0, z.data_ptr(), f.data_ptr(), 0.6, 1e-6, st) == EINVAL
    assert L.boatper_update(h, 4, z.data_ptr(), f.data_ptr(), -0.5, 1e-6, st) == EINVAL
    assert L.boatper_update(h, 4, z.data_ptr(), f.data_ptr(), 0.6, 0.0, st) == EINVAL
    empty = S.PrioritizedReplayBuffer(64, (11,), 1, precision="fp32", device=0, as_torch=True)
    assert L.boatper_sample(empty._p, 4, 0, 0, 0.4, z.data_ptr(), f.data_ptr(), st) == EINVAL
    assert L.boatper_update(empty._p, 4, z.data_ptr(), f.data_ptr(), 0.6, 1e-6, st) == EINVAL
    mem.close()
    empty.close()


@gpu
def test_device_descent_clamps_targets_on_and_past_the_edges():
    """Targets that rounding puts on or past an edge -- the total, past it, past a block's sum, on every prefix
    boundary -- on a ring with a zero tail and a total that is not exactly representable: the device returns what the
    reference returns, and never a slot of zero priority or beyond the filled ones."""
    n, filled = 3 * FAN + 100, 2 * FAN + 52
    mem = S.PrioritizedReplayBuffer(n, (11,), 1, precision="fp32", device=0, as_torch=True)
    set_mem_cntr(mem, filled)
    pr = (np.random.default_rng(5).random(filled) * 3 + 0.1).astype(np.float32)
    pr[[0, 31, 1023, 1024, 2047]] = 0   # zero leaves at chunk and block edges inside the filled range
    leaves = torch.from_numpy(pr).cuda()
    one = torch.ones(1, device="cuda")
    _lib.check(mem._L.boatper_load(mem._p, leaves.data_ptr(), filled, one.data_ptr(), filled, mem._stream()),
               "boatper_load")
    mem._filled = filled
    T = RefTree(n)
    T.levels[0][:filled] = pr
    T.resum()
    top = mem.tree_levels() - 1
    total = mem.tree_level(top).item()
    assert total == T.levels[-1][0] and float(np.float32(total)) != total
    cum = np.cumsum(pr.astype(np.float64))
    t = np.concatenate([[total, np.nextafter(total, np.inf), total * (1 + 1e-12), 2 * total],
                        T.levels[1][:2] * (1 + 1e-15), np.cumsum(T.levels[1][:2]),
                        cum, np.nextafter(cum, np.inf), np.nextafter(cum, -np.inf), [0.0]])
    got = mem.find(t).cpu().numpy()
    assert np.array_equal(got, T.descend(t.copy()))
    assert (got < filled).all() and (pr[got] > 0).all()
    assert (got[:4] == np.flatnonzero(pr)[-1]).all()
    mem.close()


@gpu
def test_sampler_frequencies_follow_the_priorities():
    """10^6 draws from a skewed 4096-slot ring: chi-square of the slot counts against p_i / sum p (fixed seed)."""
    from scipy.stats import chi2
    n = 4096
    mem = S.PrioritizedReplayBuffer(n, (11,), 1, precision="fp32", device=0, seed=1, as_torch=True, alpha=1.0,
                                    eps=1e-6)
    set_mem_cntr(mem, n)
    mem.sample_buffer(128)
    p = np.random.default_rng(0).pareto(1.5, n).astype(np.float32) + 0.01
    mem.update_priorities(torch.arange(n, device="cuda"), torch.from_numpy(p).cuda())
    counts = torch.zeros(n, dtype=torch.int64, device="cuda")
    for _ in range(250):
        idx = mem.sample_buffer(4000, beta=0.4)[5]
        counts += torch.bincount(idx, minlength=n)
    pr = mem.tree_level(0).double().cpu().numpy()
    expect = pr / pr.sum() * 1_000_000
    stat = float((((counts.cpu().numpy() - expect) ** 2) / expect).sum())
    assert stat < chi2.ppf(0.999, n - 1), stat
    mem.close()


# ---- GPU: the prioritized fused learner --------------------------------------------------------------------------------

def _agent(B, algo, learner, prioritized, seed=0):
    cfg = S.load_config(agent__batch_size=B)
    cls = S.PrioritizedReplayBuffer if prioritized else S.ReplayBuffer
    mem = cls(8192, (11,), 1, precision="fp32", device=0, as_torch=True)
    torch.manual_seed(seed)
    return ContinuousAgent(cfg, None, (11,), _env_stub(), device=0, memory=mem, learner_precision=learner,
                           algorithm=algo, prioritized=prioritized)


def _gpu_batch(B, seed):
    return {k: v.cuda() for k, v in _cpu_batch(B, seed).items()}


def _set_batch(agent, b, w=None):
    for dst, k in zip(agent._batch, ("state", "action", "reward", "new_state", "done")):
        dst.copy_(b[k].reshape(dst.shape))
    agent._eps.copy_(b["eps"])
    if w is not None:
        agent._weights.copy_(w)


def _state(agent):
    L, o = agent.learner, agent.learner.optimizer
    return ([p.detach().clone() for net in L.networks() for p in net.parameters()] +
            [p.grad.clone() for p in o.params] + [t.clone() for t in o.state_tensors()] +
            [torch.stack([x.detach().clone() for x in agent._losses])])


@gpu
@pytest.mark.parametrize("algo", ["sac1", "sac2"])
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_fused_unit_weights_equal_the_plain_fused_update(algo, B):
    b = _gpu_batch(B, B + 1)
    plain, per = _agent(B, algo, "tcgen05", False), _agent(B, algo, "tcgen05", True)
    ref = _agent(B, algo, "fp32", True)
    for a in (plain, per, ref):
        _set_batch(a, b, torch.ones(B, device="cuda") if a.prioritized else None)
        a._run_update()
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(_state(plain), _state(per)))
    td, td_ref = per._td, ref._td
    assert (td - td_ref).abs().max().item() <= 2e-3 * td_ref.abs().max().item() + 1e-5


def _weighted_emulation(agent, b, w, algo):
    """The fused update with importance weights: the unweighted bf16 emulation for the actor, value and temperature,
    and its critic pass with each row's output gradient w_i (q_i - target_i) / B.  Returns (grads, the three losses with
    the weighted critic loss, the unweighted critic loss, the rows' TD errors)."""
    L = agent.learner
    nets = [n for n in ("actor", "critic_1", "critic_2", "value", "target_value", "target_critic_1", "target_critic_2")
            if hasattr(L, n)]
    P = {n: {k: p.detach().clone() for k, p in getattr(L, n).named_parameters()} for n in nets}
    B = b["state"].shape[0]
    if algo == "sac2":
        la = L.temperature.log_alpha.detach().clone()
        grads, losses = emulate_update_sac2(P, la, b, L.gamma, L.scale, L.target_entropy)
    else:
        grads, losses = emulate_update(P, b["state"], b["action"], b["reward"], b["new_state"], b["done"], b["eps"],
                                  L.gamma, L.scale)
    r = lambda t: t.to(torch.bfloat16).float()  # noqa: E731
    heads = {"actor": ("mean", "std"), "value": ("v",), "target_value": ("v",)}

    def fwd(n, x):
        p = P[n]
        h1 = torch.relu(r(x) @ r(p["fc1.weight"]).T + p["fc1.bias"])
        h1b = r(h1)
        h2 = torch.relu(h1b @ r(p["fc2.weight"]).T + p["fc2.bias"])
        return dict(x=x, h1=h1, h1b=h1b, h2=h2,
                    y=[h2 @ p[h + ".weight"][0] + p[h + ".bias"][0] for h in heads.get(n, ("q",))])

    def bwd(n, f, dy):
        p = P[n]
        dz2 = dy[:, None] * p["q.weight"][0][None, :] * (f["h2"] > 0)
        dz1 = (r(dz2) @ r(p["fc2.weight"])) * (f["h1"] > 0)
        return {"fc1.weight": dz1.T @ f["x"], "fc1.bias": dz1.sum(0), "fc2.weight": r(dz2).T @ f["h1b"],
                "fc2.bias": dz2.sum(0), "q.weight": (dy[:, None] * f["h2"]).sum(0)[None], "q.bias": dy.sum()[None]}
    s, s2, done, e = b["state"], b["new_state"], b["done"], b["eps"].reshape(2, B)
    if algo == "sac2":
        alpha = torch.exp(la)[0]
        a_next, lp_next = _gauss_fwd(*fwd("actor", s2)["y"], e[0], 1.0)
        qt = [fwd(t, torch.cat([s2, a_next[:, None]], 1))["y"][0] for t in ("target_critic_1", "target_critic_2")]
        v = torch.minimum(qt[0], qt[1]) - alpha * lp_next
    else:
        v = fwd("target_value", s2)["y"][0]
    target = L.scale * b["reward"] + L.gamma * torch.where(done, torch.zeros_like(v), v)
    err = []
    for n in ("critic_1", "critic_2"):
        fs = fwd(n, torch.cat([s, b["action"].reshape(B, 1)], 1))
        err.append(fs["y"][0] - target)
        grads[n] = bwd(n, fs, err[-1] * w / B)
    weighted = 0.5 * (w * err[0] ** 2).mean() + 0.5 * (w * err[1] ** 2).mean()
    td = 0.5 * (err[0].abs() + err[1].abs())
    return grads, torch.stack([losses[0], losses[1], weighted]), losses[2], td


@gpu
@pytest.mark.parametrize("algo", ["sac1", "sac2"])
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_fused_weighted_update_matches_the_weighted_emulation(algo, B):
    b = _gpu_batch(B, 2 * B + 3)
    w = torch.rand(B, generator=torch.Generator().manual_seed(B)).cuda() * 0.95 + 0.05
    agent = _agent(B, algo, "tcgen05", True, seed=4)
    grads, losses, unweighted, td = _weighted_emulation(agent, b, w, algo)
    _set_batch(agent, b, w)
    agent._run_update()
    torch.cuda.synchronize()
    for n in ("actor", "critic_1", "critic_2") + (("value",) if algo == "sac1" else ()):
        for k, p in getattr(agent.learner, n).named_parameters():
            ref = grads[n][k]
            err = (p.grad - ref).abs().max().item() / max(ref.abs().max().item(), 1e-12)
            assert err <= 3e-4, (n, k, err)
    # the losses, the critic loss from the weighted partials: the weighting moves it far outside the tolerance
    got = torch.stack([x.detach() for x in agent._losses])
    assert torch.allclose(got, losses, rtol=2e-3, atol=1e-6), (got, losses)
    assert abs(losses[2].item() - unweighted.item()) > 0.05 * abs(losses[2].item())
    assert (agent._td - td).abs().max().item() <= 2e-3 * td.abs().max().item() + 1e-5


@gpu
@pytest.mark.parametrize("algo", ["sac1", "sac2"])
def test_fp32_graph_weighted_update_is_the_eager_update(algo):
    B = 512
    b = _gpu_batch(B, 11)
    w = torch.rand(B, generator=torch.Generator().manual_seed(2)).cuda() + 0.1
    graph, eager = _agent(B, algo, "fp32", True, seed=2), _agent(B, algo, "fp32", True, seed=2)
    eager.use_cuda_graph = False
    for _ in range(3):
        for a in (graph, eager):
            _set_batch(a, b, w)
            a._run_update()
        torch.cuda.synchronize()
        assert all(torch.equal(x, y) for x, y in zip(_state(graph), _state(eager)))
        assert torch.equal(graph._td, eager._td)


# ---- GPU: the loop ----------------------------------------------------------------------------------------------------

def _loop_agent(algo, learner, tmp, seed=3):
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
    env = S.BatchedBoatEnv(cfg, 2048, seed=seed, precision="fp32", device=0, auto_reset=True)
    torch.manual_seed(seed)
    agent = ContinuousAgent(cfg, str(tmp), (11,), env, device=0, seed=seed, learner_precision=learner,
                            policy_precision="tcgen05", algorithm=algo, prioritized=True, priority_alpha=0.7,
                            priority_beta=0.5, priority_beta_updates=20)
    return env, agent


def _run(env, agent, iters, collect=True):
    out = []
    for _ in range(iters):
        if collect:
            agent.collect(env, 2)
        else:
            agent.step_and_remember(env, agent.choose_action(env.obs).squeeze(-1))
        losses = agent.learn()
        if losses is not None:
            out.append(torch.stack([x.detach().clone() for x in losses]))
    return out


@gpu
@pytest.mark.parametrize("collect", [True, False])
def test_prioritized_learn_is_bit_reproducible(collect, tmp_path):
    runs = []
    for _ in range(2):
        env, agent = _loop_agent("sac1", "tcgen05", tmp_path)
        env.reset()
        losses = _run(env, agent, 8, collect)
        runs.append((losses, _state(agent), agent.memory.tree_level(0).clone(), agent._idx.clone()))
        agent.memory.close()
        env.close()
    (la, sa, pa, ia), (lb, sb, pb, ib) = runs
    assert len(la) > 0 and all(torch.equal(x, y) for x, y in zip(la + sa, lb + sb))
    assert torch.equal(pa, pb) and torch.equal(ia, ib)


@gpu
@pytest.mark.parametrize("algo,learner", [("sac1", "fp32"), ("sac1", "tcgen05"), ("sac2", "fp32"), ("sac2", "tcgen05")])
def test_prioritized_whole_loop_checkpoint_resume_is_exact(algo, learner, tmp_path):
    env, agent = _loop_agent(algo, learner, tmp_path)
    env.reset()
    _run(env, agent, 8)
    torch.save({"env": env.state_dict(), "agent": agent.state_dict()}, tmp_path / "full.pt")
    acting = agent.tensor_core_policy().steps
    tail_a = _run(env, agent, 5)
    snap_a, mem_a = _state(agent), agent.memory.state_dict()
    env2, agent2 = _loop_agent(algo, learner, tmp_path, seed=3)
    ck = torch.load(tmp_path / "full.pt", weights_only=False)
    env2.load_state_dict(ck["env"])
    agent2.load_state_dict(ck["agent"])
    agent2.tensor_core_policy().steps = acting
    tail_b = _run(env2, agent2, 5)
    assert all(torch.equal(x, y) for x, y in zip(tail_a + snap_a, tail_b + _state(agent2)))
    mem_b = agent2.memory.state_dict()
    assert "priorities" in mem_a
    for k, v in mem_a.items():
        assert (torch.equal(v, mem_b[k]) if isinstance(v, torch.Tensor) else v == mem_b[k]), k
    assert abs(agent2.priority_beta() - (0.5 + 0.5 * min(1.0, agent2.updates / 20))) < 1e-12
    for x in (env, env2, agent.memory, agent2.memory):
        x.close()


@gpu
@pytest.mark.parametrize("algo", ["sac1", "sac2"])
def test_train_sac_prioritized_end_to_end(algo, capsys):
    import train_sac
    flags = ["--envs", "1024", "--iters", "6", "--warmup-iters", "2", "--log-every", "2", "--experiment", "6",
             "--buffer", "100000", "--policy-precision", "tcgen05", "--collect-steps", "4", "--updates-per-iter", "2",
             "--set", "agent__batch_size=256", "--learner-precision", "tcgen05", "--algorithm", algo,
             "--prioritized", "--priority-alpha", "0.5", "--priority-beta-updates", "10"]
    train_sac.main(flags)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["prioritized"] is True and line["priority_alpha"] == 0.5 and line["priority_beta"] == 0.4
    assert line["priority_beta_updates"] == 10 and line["priority_eps"] == 1e-6
    losses = line.get("losses_v_pi_q") or line.get("losses_t_pi_q")
    assert losses is None or all(math.isfinite(x) for x in losses)
