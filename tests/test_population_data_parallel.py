"""Data-parallel population training (AgentPopulation(data_parallel=...), boatagent_sac_gradients_members,
boatagent_adam_polyak_members, train_sac --population P --data-parallel): the split member launches against the fused
member update and the per-agent launches, bit for bit; a one-rank group against the plain population; two ranks
sharing one GPU over gloo against a one-process emulation of the averaged updates; the driver's rejections."""
import ctypes as C
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))

import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200 import _lib  # noqa: E402

EINVAL = -1
gpu = pytest.mark.gpu
TWO_GPUS = pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2,
                              reason="needs two visible GPUs")
BASE = ["--policy-precision", "tcgen05", "--learner-precision", "tcgen05", "--collect-steps", "8"]


# ---- CPU ------------------------------------------------------------------------------------------------------------

def _world(monkeypatch, n):
    monkeypatch.setenv("WORLD_SIZE", str(n))
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("LOCAL_RANK", "0")
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("CUDA work before the flags were checked"))


@pytest.mark.parametrize("world, flags", [
    (2, ["--population", "4", "--data-parallel", "--envs", "1001"]),          # envs do not split over the ranks
    (1, ["--population", "4", "--data-parallel"]),                            # a one-rank group is plain --population
    (2, ["--population", "4", "--pbt-every", "5"]),                           # rounds across ranks need --data-parallel
    (2, ["--population", "4", "--data-parallel", "--overlap"]),
    (2, ["--population", "4", "--data-parallel", "--record-envs", "2", "--experiments-root", "/nonexistent"]),
    (2, ["--data-parallel", "--tune"]),                                       # no population: one agent, no draws
    (2, ["--data-parallel", "--pbt-every", "5"]),
])
def test_driver_rejects_before_cuda_work(world, flags, monkeypatch):
    import train_sac
    _world(monkeypatch, world)
    with pytest.raises(SystemExit) as e:
        train_sac.main(BASE + flags)
    assert e.value.code == 2


def _fake_slots(bad=None):
    """A 26-slot table with the agent's shapes and dummy (never dereferenced) pointers; `bad` corrupts one field."""
    from sac_agent_b200.continuous_agent import _AdamSlot
    numel = [2816, 256, 65536, 256, 256, 1, 256, 1] + [3072, 256, 65536, 256, 256, 1] * 2 + [2816, 256, 65536, 256,
                                                                                              256, 1]
    slots = (_AdamSlot * 26)()
    for k, n in enumerate(numel):
        slots[k] = _AdamSlot(256, 512, 768, 1024, 1280 if k >= 20 else None, n, 1e-3, 0)
    if bad is not None:
        k, field, value = bad
        setattr(slots[k], field, value)
    return slots


def _fake_member(slots, adam_state=2048, n_slots=26):
    return _lib.SacMember(16, 16, 16, 16, 16, 16, 16, C.cast(slots, C.c_void_p), n_slots, 0.99, 1.0, 0.005,
                          adam_state, 16)


def test_member_split_abi_rejects_bad_tables_without_launching():
    L = S.lib()
    launches = L.boatenv_kernel_launches()
    tbl = (_lib.SacMember * 17)()
    ws = C.c_void_p(16)
    # gradients: the checks of boatagent_sac_update_members
    for n in (0, 17, -1):
        assert L.boatagent_sac_gradients_members(tbl, n, 1024, 0.5, ws, 1 << 40, None) == EINVAL
    assert L.boatagent_sac_gradients_members(None, 1, 1024, 0.5, ws, 1 << 40, None) == EINVAL
    assert L.boatagent_sac_gradients_members(tbl, 1, 1000, 0.5, ws, 1 << 40, None) == EINVAL   # batch % 128
    assert L.boatagent_sac_gradients_members(tbl, 1, 1024, 0.5, None, 1 << 40, None) == EINVAL
    assert L.boatagent_sac_gradients_members(tbl, 1, 1024, 0.5, ws, 1 << 40, None) == EINVAL   # NULL members
    one = (_lib.SacMember * 1)(_fake_member(_fake_slots()))
    assert L.boatagent_sac_gradients_members(one, 1, 1024, 0.5, ws, 16, None) == EINVAL         # workspace too small
    # Adam: the table's slots and state
    for n in (0, 17, -1):
        assert L.boatagent_adam_polyak_members(tbl, n, 0.9, 0.999, 1e-8, None) == EINVAL
    assert L.boatagent_adam_polyak_members(None, 1, 0.9, 0.999, 1e-8, None) == EINVAL
    assert L.boatagent_adam_polyak_members(tbl, 1, 0.9, 0.999, 1e-8, None) == EINVAL            # NULL members
    keep = []
    for bad in [(2, "numel", 65535), (20, "target", None), (3, "target", 4096), (5, "param", None),
                (5, "grad", None), (7, "exp_avg", None), (25, "exp_avg_sq", None)]:
        slots = _fake_slots(bad)
        keep.append(slots)
        two = (_lib.SacMember * 2)(_fake_member(_fake_slots()), _fake_member(slots))   # the second member is bad
        assert L.boatagent_adam_polyak_members(two, 2, 0.9, 0.999, 1e-8, None) == EINVAL, bad
    good = _fake_slots()
    for member in (_fake_member(good, adam_state=None), _fake_member(good, n_slots=25), _fake_member(None)):
        assert L.boatagent_adam_polyak_members((_lib.SacMember * 1)(member), 1, 0.9, 0.999, 1e-8, None) == EINVAL
    assert L.boatenv_kernel_launches() == launches


# ---- GPU: the kernels -----------------------------------------------------------------------------------------------

def _learner(seed, k):
    """A learner with member k's hyper-parameters (learning rates, gamma, tau, reward scale all differ)."""
    from sac_agent_b200.continuous_agent import SACLearner
    torch.manual_seed(seed)
    L = SACLearner((11,), 1, np.ones(1, dtype=np.float32), 3e-4, 3e-4, 0.99, 0.005, 10.0, device="cuda")
    o = L.optimizer
    for i, p in enumerate(o.params):
        o._slots[i].lr = (3e-4 if i < 8 else 5e-4) * (1.0 + 0.37 * k)
        p.grad = torch.zeros_like(p)
        o._slots[i].grad = p.grad.data_ptr()
    L.gamma = 0.99 - 0.01 * k
    L.tau = o.tau = 0.005 * (1 + k)
    L.scale = 10.0 + k
    return L


def _inputs(B, k, it):
    g = torch.Generator(device="cuda").manual_seed(1000 * it + k)
    kw = dict(device="cuda", generator=g)
    return (torch.rand((B, 11), **kw), torch.rand((B, 1), **kw) * 2 - 1, torch.randn(B, **kw),
            torch.rand((B, 11), **kw), (torch.rand(B, **kw) < 0.1).to(torch.uint8), torch.randn((2, B, 1), **kw))


def _entry(L, inp, losses):
    o = L.optimizer
    s, a, r, s2, d, eps = inp
    return _lib.SacMember(s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), eps.data_ptr(),
                          L.actor.max_action.data_ptr(), C.cast(o._slots, C.c_void_p), len(o.params), float(L.gamma),
                          float(L.scale), float(o.tau), o.state.data_ptr(), losses.data_ptr())


def _state(L, losses):
    o = L.optimizer
    return ([p.detach().clone() for net in L.networks() for p in net.parameters()]
            + [p.grad.clone() for p in o.params] + [t.clone() for t in o.state_tensors()] + [losses.clone()])


def _same(a, b, what):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), f"{what}: tensor {i} differs"


@gpu
@pytest.mark.parametrize("P", [1, 3, 16])
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_split_member_launches_are_the_fused_and_the_solo_launches(P, B):
    """Over three updates: gradients_members(1) + adam_polyak_members == sac_update_members; gradients_members(s) ==
    P boatagent_sac_gradients(s); adam_polyak_members == P boatagent_adam_polyak_step.  All bit for bit."""
    Lib = S.lib()
    fused = [_learner(10 + k, k) for k in range(P)]      # boatagent_sac_update_members
    split = [_learner(10 + k, k) for k in range(P)]      # gradients_members(1) + adam_polyak_members
    solo = [_learner(10 + k, k) for k in range(P)]       # split's gradients, stepped by boatagent_adam_polyak_step
    lf, ls, lo = ([torch.zeros(3, device="cuda") for _ in range(P)] for _ in range(3))
    slice_bytes = int(Lib.boatagent_sac_update_workspace_bytes(B))
    ws = torch.empty(P * slice_bytes, dtype=torch.uint8, device="cuda")
    ws1 = torch.empty(slice_bytes, dtype=torch.uint8, device="cuda")
    o0 = fused[0].optimizer
    for it in range(3):
        inps = [_inputs(B, k, it) for k in range(P)]
        tf = (_lib.SacMember * P)(*[_entry(L, i, l) for L, i, l in zip(fused, inps, lf)])
        ts = (_lib.SacMember * P)(*[_entry(L, i, l) for L, i, l in zip(split, inps, ls)])
        assert Lib.boatagent_sac_update_members(tf, P, B, o0.betas[0], o0.betas[1], o0.eps, ws.data_ptr(), ws.numel(),
                                                None) == 0

        # gradients_members(s) against P solo gradients(s) on split's current weights (nothing else is written)
        scale = 0.25
        before = [_state(L, l) for L, l in zip(split, ls)]
        assert Lib.boatagent_sac_gradients_members(ts, P, B, scale, ws.data_ptr(), ws.numel(), None) == 0
        torch.cuda.synchronize()
        got = [_state(L, l) for L, l in zip(split, ls)]
        for k, (L, inp) in enumerate(zip(split, inps)):
            o, (s, a, r, s2, d, eps) = L.optimizer, inp
            grads = [torch.zeros_like(p) for p in o.params]
            for i, g in enumerate(grads):
                o._slots[i].grad = g.data_ptr()
            loss = torch.zeros(3, device="cuda")
            assert Lib.boatagent_sac_gradients(
                s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), eps.data_ptr(),
                L.actor.max_action.data_ptr(), B, float(L.gamma), float(L.scale), o._slots, len(o.params), scale,
                loss.data_ptr(), ws1.data_ptr(), ws1.numel(), None) == 0
            for i, p in enumerate(o.params):
                o._slots[i].grad = p.grad.data_ptr()
            torch.cuda.synchronize()
            n = len(grads)
            _same(got[k][:32], before[k][:32], f"P={P} B={B} it={it} member {k}: weights untouched")
            _same(got[k][32:32 + n], grads, f"P={P} B={B} it={it} member {k}: scaled gradients")
            _same(got[k][32 + n:-1], before[k][32 + n:-1], f"member {k}: Adam state untouched")
            assert torch.equal(got[k][-1], loss), (P, B, it, k)

        # the update of split: gradients_members(1) + adam_polyak_members; solo: the same gradients, P Adam steps
        assert Lib.boatagent_sac_gradients_members(ts, P, B, 1.0, ws.data_ptr(), ws.numel(), None) == 0
        for Ls, Lo in zip(split, solo):
            for p, q in zip(Ls.optimizer.params, Lo.optimizer.params):
                q.grad.copy_(p.grad)
        assert Lib.boatagent_adam_polyak_members(ts, P, o0.betas[0], o0.betas[1], o0.eps, None) == 0
        for L in solo:
            o = L.optimizer
            assert Lib.boatagent_adam_polyak_step(o._slots, len(o.params), o.betas[0], o.betas[1], o.eps, o.tau,
                                                  o.state.data_ptr(), None) == 0
        torch.cuda.synchronize()
        for k in range(P):
            _same(_state(fused[k], lf[k]), _state(split[k], ls[k]), f"P={P} B={B} it={it} member {k}: split vs fused")
            _same(_state(split[k], ls[k])[:-1], _state(solo[k], lo[k])[:-1], f"member {k}: Adam members vs solo")
    assert all(int(L.optimizer.state[0]) == 3 for L in split + solo)


# ---- GPU: one rank --------------------------------------------------------------------------------------------------

@pytest.fixture
def gloo_world_1(tmp_path):
    """A one-rank gloo default group (file-store rendezvous), destroyed after the test."""
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/store", rank=0, world_size=1)
    yield dist.group.WORLD
    dist.destroy_process_group()


def _member_state(a):
    o = a.learner.optimizer
    sd = a.memory.state_dict()
    return ([p.detach().clone() for net in a.learner.networks() for p in net.parameters()]
            + [p.grad.clone() for p in o.params] + [t.clone() for t in o.state_tensors()] + [a._loss_buf.clone()]
            + [sd[k] for k in ("state", "action", "reward", "new_state", "terminal")])


def _population_run(data_parallel, P=3, rounds=6):
    cfg = S.load_config(base_settings__experiment=5, agent__batch_size=256)
    torch.manual_seed(7)
    pop = S.AgentPopulation(cfg, P, 512, seed=4, buffer_size=16384, data_parallel=data_parallel)
    pop.reset()
    losses = []
    for r in range(rounds):
        pop.collect(2)
        for _ in range(2):
            out = pop.learn()
            if out is not None:
                losses.append(torch.stack([torch.stack(x) for x in out]).clone())
        if r == 3:
            pop.exploit_explore([c["return_sum"] / max(c["episodes"], 1.0) for c in pop.counters()], random.Random(2))
    torch.cuda.synchronize()
    out = (losses, [_member_state(a) for a in pop.members], [env.obs.clone() for env in pop.envs], pop.counters(),
           [a.hyperparameters() for a in pop.members], [a.memory.mem_cntr for a in pop.members])
    pop.close()
    return out


@gpu
def test_one_rank_group_is_the_plain_population(gloo_world_1):
    plain = _population_run(None)
    dp = _population_run(gloo_world_1)
    assert len(plain[0]) == len(dp[0]) >= 8
    _same(plain[0], dp[0], "losses")
    for m, (a, b) in enumerate(zip(plain[1], dp[1])):
        _same(a, b, f"member {m}: weights, gradients, Adam state, losses, ring")
    _same(plain[2], dp[2], "observations")
    assert plain[3:] == dp[3:]


def _tree(root):
    """{relative path with the member's directory name reduced to its member index: file bytes}, timestamps dropped."""
    import re
    out = {}
    for d, _, files in os.walk(root):
        for f in files:
            rel = os.path.relpath(os.path.join(d, f), root)
            key = re.sub(r"experiment_(r0_)?m(\d+)_[0-9_-]+", r"m\2", rel)
            data = open(os.path.join(d, f), "rb").read()
            if f == "overview.csv":
                data = re.sub(rb"experiment_(r0_)?m(\d+)_[0-9_-]+", rb"m\2", data)
            out[key] = data
    return out


@gpu
def test_driver_population_function_with_a_one_rank_group(gloo_world_1, tmp_path, monkeypatch):
    import train_sac
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    common = BASE[:4] + ["--collect-steps", "2", "--population", "3", "--envs", "1024", "--iters", "20",
                         "--warmup-iters", "2", "--buffer", "20000", "--set", "agent__batch_size=256", "--log-every",
                         "5", "--tune", "--pbt-every", "5"]
    torch.cuda.set_device(0)
    plain = train_sac.main(common + ["--experiments-root", str(tmp_path / "plain")])
    import argparse
    args = argparse.Namespace(**_parsed(train_sac, common + ["--experiments-root", str(tmp_path / "dp")]))
    dp = train_sac.train_population(args, 0, 0, 1, group=gloo_world_1)
    assert dp["data_parallel"] is True and dp["effective_batch"] == 256 and "data_parallel" not in plain
    for k in ("losses_v_pi_q", "episodes", "reached_goal", "hpsets", "hyperparameters", "pbt_adoptions", "members"):
        assert dp[k] == plain[k], k
    assert _tree(tmp_path / "plain") == _tree(tmp_path / "dp")


def _parsed(train_sac, argv):
    """The driver's parsed arguments for argv (main() with train_population intercepted)."""
    got = {}

    def grab(args, *a, **kw):
        got.update(vars(args))
        return None
    keep = train_sac.train_population
    train_sac.train_population = grab
    try:
        train_sac.main(argv)
    finally:
        train_sac.train_population = keep
    return got


# ---- two ranks ------------------------------------------------------------------------------------------------------
_WORKER = r"""
import os, random, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
import sac_agent_b200 as S
rank, local_rank, world = S.sharding.dist_info()
torch.cuda.set_device(local_rank)
backend, out_dir = sys.argv[1], sys.argv[2]
dist.init_process_group(backend, init_method="file://" + out_dir + "/store", rank=rank, world_size=world)
cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
try:
    S.AgentPopulation(cfg, 2, 256 + 128 * rank, seed=1, buffer_size=4096, data_parallel=True)
    raise SystemExit("unequal populations were accepted")
except ValueError:
    pass
torch.manual_seed(50 + rank)               # each rank its own Gaussian draws
pop = S.AgentPopulation(cfg, 3, 512, seed=1, buffer_size=16384, data_parallel=True)
assert pop.rank == rank and [e.env_id_offset for e in pop.envs] == [(m * world + rank) * 512 for m in range(3)]
pop.reset()
def snap():
    return [[t.cpu().clone() for t in a.training_tensors()] for a in pop.members], [a.hyperparameters() for a in pop.members]
rec = dict(segments=[], final=None)
seg = dict(start=snap(), batches=[], eps=[], losses=[])
for r in range(8):
    pop.collect(2)
    for _ in range(2):
        out = pop.learn()
        if out is not None:
            seg["batches"].append([[t.cpu().clone() for t in a._batch] for a in pop.members])
            seg["eps"].append([a._eps.cpu().clone() for a in pop.members])
            seg["losses"].append([torch.stack(x).cpu().clone() for x in out])
    if r == 4:                             # a population round from the summed counters, the same rng everywhere
        c = pop.counters()
        scores = [x["episodes"] - (1e9 if m == 1 else 0.0) for m, x in enumerate(c)]   # member 1 adopts
        rec["round"] = pop.exploit_explore(scores, random.Random(9))
        rec["segments"].append(seg)
        seg = dict(start=snap(), batches=[], eps=[], losses=[])
rec["segments"].append(seg)
torch.cuda.synchronize()
rec["final"] = snap()
rec["rings"] = [a.memory.state_dict()["state"].cpu().clone() for a in pop.members]
torch.save(rec, os.path.join(out_dir, f"rank{{rank}}.pt"))
dist.barrier()
pop.close()
dist.destroy_process_group()
print("DP_OK")
"""


def _two_ranks(tmp_path, backend):
    script = tmp_path / "pop_worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r if backend == "nccl" else 0))
        procs.append(subprocess.Popen([sys.executable, str(script), backend, str(tmp_path)], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    for p in procs:
        out, err = p.communicate(timeout=900)
        assert p.returncode == 0 and "DP_OK" in out, err[-3000:]
    return [torch.load(tmp_path / f"rank{r}.pt", weights_only=False) for r in range(2)]


def _emulate(seg0, seg1, m):
    """Member m over one segment in one process: from its recorded start, each update is DeviceAdam on
    0.5 g0 + 0.5 g1, g_r the boatagent_sac_gradients of rank r's recorded batch and draws.  Returns (mean losses
    per update, training tensors at the end)."""
    from sac_agent_b200.continuous_agent import ContinuousAgent
    mem = S.ReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    env = type("E", (), {"action_space": S.Box(low=-1, high=1, dtype=np.float32)})()
    agent = ContinuousAgent(S.load_config(base_settings__experiment=6, agent__batch_size=256), None, (11,), env,
                            device=0, memory=mem, learner_precision="tcgen05")
    agent.set_hyperparameters(**seg0["start"][1][m])
    with torch.no_grad():
        for t, v in zip(agent.training_tensors(), seg0["start"][0][m]):
            t.copy_(v)
    L, o = agent.learner, agent.learner.optimizer
    losses = []
    for it in range(len(seg0["batches"])):
        per_rank = []
        for seg in (seg0, seg1):
            for t, v in zip(agent._batch, seg["batches"][it][m]):
                t.copy_(v)
            agent._eps.copy_(seg["eps"][it][m])
            g = [torch.zeros_like(p) for p in o.params]
            lv = torch.zeros(3, device="cuda")
            for k, x in enumerate(g):
                o._slots[k].grad = x.data_ptr()
            s, a, r, s2, d = agent._batch
            assert o._L.boatagent_sac_gradients(
                s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), agent._eps.data_ptr(),
                L.actor.max_action.data_ptr(), 256, float(L.gamma), float(L.scale), o._slots, len(o.params), 1.0,
                lv.data_ptr(), agent._ws.data_ptr(), agent._ws.numel(), None) == 0
            per_rank.append((g, lv))
        (g0, l0), (g1, l1) = per_rank
        o.step([0.5 * a + 0.5 * b for a, b in zip(g0, g1)])
        losses.append(0.5 * l0 + 0.5 * l1)
    torch.cuda.synchronize()
    out = [l.cpu() for l in losses], [t.cpu().clone() for t in agent.training_tensors()]
    mem.close()
    return out


def _check_two_ranks(recs):
    rec0, rec1 = recs
    assert rec0["round"]["adopted"] and rec0["round"] == rec1["round"]
    for m in range(3):
        for a, b in zip(rec0["final"][0][m], rec1["final"][0][m]):   # weights, target, Adam moments, step counter
            assert torch.equal(a, b), m
        assert rec0["final"][1][m] == rec1["final"][1][m]
        assert not torch.equal(rec0["rings"][m], rec1["rings"][m])   # each rank its own ring
    for i, (s0, s1) in enumerate(zip(rec0["segments"], rec1["segments"])):
        assert len(s0["batches"]) == len(s1["batches"]) > 0
        for m in range(3):
            end = rec0["segments"][i + 1]["start"][0][m] if i + 1 < len(rec0["segments"]) else None
            losses, state = _emulate(s0, s1, m)
            for it, l in enumerate(losses):
                assert torch.equal(s0["losses"][it][m], l) and torch.equal(s1["losses"][it][m], l), (i, m, it)
            if end is None:
                end = rec0["final"][0][m]
            elif m in rec0["round"]["adopted"]:   # the round overwrote this member: check its state before it
                continue
            for a, b in zip(state, end):
                assert torch.equal(a, b), (i, m)


@gpu
def test_two_ranks_share_one_gpu_over_gloo(tmp_path):
    _check_two_ranks(_two_ranks(tmp_path, "gloo"))


@gpu
@TWO_GPUS
def test_two_ranks_over_nccl(tmp_path):
    _check_two_ranks(_two_ranks(tmp_path, "nccl"))


@gpu
@TWO_GPUS
def test_driver_two_ranks_under_torchrun(tmp_path):
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "examples", "train_sac.py")] + BASE[:4] +
                       ["--collect-steps", "2", "--population", "3", "--data-parallel", "--tune", "--pbt-every", "5",
                        "--envs", "2048", "--iters", "20", "--warmup-iters", "2", "--buffer", "20000", "--set",
                        "agent__batch_size=256", "--experiments-root", str(tmp_path), "--log-every", "5"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    assert summary["data_parallel"] is True and summary["effective_batch"] == 512 and summary["members"] == 3
    assert sorted(d.split("_")[1] for d in os.listdir(os.path.join(tmp_path, "setting_5")) if d != "overview.csv") == \
        ["m0", "m1", "m2"]
