"""Data-parallel SAC: ContinuousAgent(data_parallel=...), boatagent_sac_gradients (csrc/learner.cu) and
train_sac.py --data-parallel.

The mode's promise is exactness: the split update (gradients, all-reduce, Adam) is the fused update bit for bit at one
rank, and at two ranks every rank holds the same bits as a single process that averages the two ranks' gradients and
applies DeviceAdam.  Two ranks share cuda:0 over gloo here (gloo all-reduces CUDA tensors through the host); the NCCL
and torchrun variants need two GPUs.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200.continuous_agent import ContinuousAgent, DataParallelState  # noqa: E402

EINVAL, EALIGN = -1, -7
TWO_GPUS = pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2,
                              reason="needs two visible GPUs")


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("extra", [["--tune"], ["--pbt-every", "10"], ["--overlap"], ["--envs", "1000"]])
def test_driver_rejects_data_parallel_combinations(extra, monkeypatch):
    """Exit code 2 from argparse, before any CUDA work (this runs without a GPU)."""
    import train_sac
    monkeypatch.setenv("WORLD_SIZE", "3")   # 1000 envs do not split over 3 ranks
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("LOCAL_RANK", "0")
    with pytest.raises(SystemExit) as e:
        train_sac.main(["--data-parallel", "--envs", "999"] + extra)
    assert e.value.code == 2


def test_learner_gradients_are_the_update_gradients():
    """SACLearner.gradients writes scale times what update() leaves in .grad, and scale times its losses."""
    from sac_agent_b200.continuous_agent import SACLearner
    torch.manual_seed(0)
    L = SACLearner((11,), 1, np.array([1.0], dtype=np.float32), 5e-3, 3e-4, 0.99, 0.005, 10.0, device="cpu",
                   torch_reference_math=True)
    g = torch.Generator().manual_seed(1)
    B = 64
    batch = (torch.rand(B, 11, generator=g), torch.rand(B, 1, generator=g), torch.randn(B, generator=g),
             torch.rand(B, 11, generator=g), torch.rand(B, generator=g) < 0.1)
    eps = torch.randn(2, B, 1, generator=g)
    params = L._actor_params + L._critic_params + L._value_params
    out = [torch.zeros_like(p) for p in params] + [torch.zeros(()) for _ in range(3)]
    L.gradients(*batch, eps[0], eps[1], out, scale=0.5)
    losses = L.update(*batch, eps_sample=eps[0], eps_rsample=eps[1])
    for o, p in zip(out, params):
        assert torch.equal(o, 0.5 * p.grad)
    for o, x in zip(out[-3:], losses):
        assert torch.equal(o, 0.5 * x)


def test_population_round_rejects_a_data_parallel_agent():
    import random
    from sac_agent_b200 import population as P
    hp = dict(alpha=0.003, beta=0.003, gamma=0.99, tau=0.005)
    with pytest.raises(ValueError):
        P.exploit_explore(DataParallelState([torch.zeros(3)]), hp, 0.0, random.Random(0))


# ---- one GPU ----------------------------------------------------------------------------------------------------------
def _env_stub():
    return type("E", (), {"action_space": S.Box(low=-1, high=1, dtype=np.float32)})()


@pytest.fixture
def gloo_world_1(tmp_path):
    """A one-rank gloo default group (file-store rendezvous), destroyed after the test."""
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/store", rank=0, world_size=1)
    yield
    dist.destroy_process_group()


def _slot_grads(agent):
    o = agent.learner.optimizer
    grads = [torch.zeros_like(p) for p in o.params]
    for k, g in enumerate(grads):
        o._slots[k].grad = g.data_ptr()
    return grads


def _sac_gradients(agent, grad_scale, loss_out, **over):
    """boatagent_sac_gradients on the agent's static batch and eps (keyword overrides for the error tests)."""
    L, o = agent.learner, agent.learner.optimizer
    s, a, r, s2, d = agent._batch
    args = dict(state=s.data_ptr(), action=a.data_ptr(), reward=r.data_ptr(), new_state=s2.data_ptr(),
                done=d.data_ptr(), eps=agent._eps.data_ptr(), max_action=L.actor.max_action.data_ptr(),
                batch=agent.batch_size, slots=o._slots, n_slots=len(o.params), losses=loss_out.data_ptr(),
                ws=agent._ws.data_ptr(), ws_bytes=agent._ws.numel())
    args.update(over)
    return o._L.boatagent_sac_gradients(args["state"], args["action"], args["reward"], args["new_state"], args["done"],
                                        args["eps"], args["max_action"], args["batch"], float(L.gamma), float(L.scale),
                                        args["slots"], args["n_slots"], grad_scale, args["losses"], args["ws"],
                                        args["ws_bytes"], None)


def _fill_batch(agent, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    B = agent.batch_size
    st = torch.rand(B, 11, generator=g) * 2 - 1
    s, a, r, s2, d = agent._batch
    s.copy_(st)
    a.copy_(torch.rand(B, 1, generator=g) * 2 - 1)
    r.copy_(torch.randn(B, generator=g))
    s2.copy_(st + 0.1 * torch.randn(B, 11, generator=g))
    d.copy_((torch.rand(B, generator=g) < 0.1).to(torch.uint8))
    agent._eps.copy_(torch.randn(2, B, 1, generator=g))


@pytest.mark.gpu
@pytest.mark.parametrize("B", [128, 1024, 4096])
def test_gradients_then_adam_is_the_fused_update(B):
    """boatagent_sac_gradients(grad_scale = 1) + boatagent_adam_polyak_step == boatagent_sac_update, bit for bit:
    gradients, weights, target, Adam moments, step counter and losses, over three consecutive updates."""
    mem = S.ReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    torch.manual_seed(1)
    fused = ContinuousAgent(S.load_config(agent__batch_size=B), None, (11,), _env_stub(), device=0, memory=mem,
                            learner_precision="tcgen05")
    torch.manual_seed(1)
    split = ContinuousAgent(S.load_config(agent__batch_size=B), None, (11,), _env_stub(), device=0, memory=mem,
                            learner_precision="tcgen05")
    grads, losses = _slot_grads(split), torch.zeros(3, device="cuda")
    for it in range(3):
        _fill_batch(fused, 10 * B + it)
        _fill_batch(split, 10 * B + it)
        got = [x.clone() for x in fused._fused_update()]
        o = split.learner.optimizer
        for k, g in enumerate(grads):
            o._slots[k].grad = g.data_ptr()
        assert _sac_gradients(split, 1.0, losses) == 0
        o.step(grads)
        torch.cuda.synchronize()
        assert torch.equal(torch.stack(got), losses), it
        for p, g in zip(fused.learner.optimizer.params, grads):
            assert torch.equal(p.grad, g)
        for x, y in zip(fused.training_tensors(), split.training_tensors()):
            assert torch.equal(x, y)
    assert int(split.learner.optimizer.state[0]) == 3
    mem.close()


@pytest.mark.gpu
def test_gradients_scale_and_errors():
    """grad_scale multiplies gradients and losses; the call leaves weights and Adam state alone; its ABI errors."""
    mem = S.ReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    agent = ContinuousAgent(S.load_config(agent__batch_size=256), None, (11,), _env_stub(), device=0, memory=mem,
                            learner_precision="tcgen05")
    _fill_batch(agent, 7)
    before = [t.clone() for t in agent.training_tensors()]
    g1 = _slot_grads(agent)
    l1 = torch.zeros(3, device="cuda")
    assert _sac_gradients(agent, 1.0, l1) == 0
    g4 = _slot_grads(agent)
    l4 = torch.zeros(3, device="cuda")
    assert _sac_gradients(agent, 0.25, l4) == 0
    torch.cuda.synchronize()
    for a, b in zip(g1, g4):
        assert torch.equal(a * 0.25, b)
    assert torch.equal(l1 * 0.25, l4)
    for x, y in zip(before, agent.training_tensors()):
        assert torch.equal(x, y)

    for name in ("state", "action", "reward", "new_state", "done", "eps", "max_action", "slots", "losses", "ws"):
        assert _sac_gradients(agent, 1.0, l1, **{name: None}) == EINVAL, name
    for bad in (0, 100, 384):   # 384: a valid batch, but larger than the workspace
        assert _sac_gradients(agent, 1.0, l1, batch=bad) == EINVAL, bad
    assert _sac_gradients(agent, 1.0, l1, n_slots=25) == EINVAL
    assert _sac_gradients(agent, 1.0, l1, ws_bytes=agent._ws.numel() - 1) == EINVAL
    assert _sac_gradients(agent, 1.0, l1, ws=agent._ws.data_ptr() + 4) == EALIGN
    o = agent.learner.optimizer
    keep = o._slots[2].numel
    o._slots[2].numel = keep - 1
    assert _sac_gradients(agent, 1.0, l1) == EINVAL
    o._slots[2].numel = keep
    keep = o._slots[20].target
    o._slots[20].target = None
    assert _sac_gradients(agent, 1.0, l1) == EINVAL
    o._slots[20].target = keep
    keep = o._slots[5].grad
    o._slots[5].grad = None
    assert _sac_gradients(agent, 1.0, l1) == EINVAL
    o._slots[5].grad = keep
    mem.close()


MODES = {"fp32-eager": dict(learner_precision="fp32", use_cuda_graph=False),
         "fp32-graph": dict(learner_precision="fp32", use_cuda_graph=True),
         "tcgen05": dict(learner_precision="tcgen05")}


def _run(mode, iters, data_parallel):
    """`iters` rounds of collect + learn at 1024 envs, from fixed seeds; (losses per round, final training tensors)."""
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
    env = S.BatchedBoatEnv(cfg, 1024, seed=3, precision="fp32", device=0, auto_reset=True)
    mem = S.ReplayBuffer(100_000, (11,), 1, precision="fp32", device=0, seed=4, as_torch=True)
    torch.manual_seed(5)
    agent = ContinuousAgent(cfg, None, (11,), env, device=0, seed=4, memory=mem, policy_precision="tcgen05",
                            data_parallel=data_parallel, **MODES[mode])
    env.reset()
    losses = []
    for _ in range(iters):
        agent.collect(env, 1)
        out = agent.learn()
        losses.append(None if out is None else torch.stack([x.clone() for x in out]))
    torch.cuda.synchronize()
    state = [t.clone() for t in agent.training_tensors()]
    env.close(); mem.close()
    return losses, state


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_world_1_is_the_plain_agent(mode, gloo_world_1):
    """A data-parallel agent on a one-rank group makes exactly the plain agent's updates."""
    plain_l, plain_s = _run(mode, 20, None)
    dp_l, dp_s = _run(mode, 20, True)
    assert sum(x is not None for x in plain_l) >= 19
    for a, b in zip(plain_l, dp_l):
        assert (a is None and b is None) or torch.equal(a, b)
    for a, b in zip(plain_s, dp_s):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_data_parallel_rejections(gloo_world_1):
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
    env = S.BatchedBoatEnv(cfg, 1024, seed=3, precision="fp32", device=0, auto_reset=True)
    mem = S.ReplayBuffer(10_000, (11,), 1, precision="fp32", device=0, as_torch=True)
    agent = ContinuousAgent(cfg, None, (11,), env, device=0, memory=mem, data_parallel=True)
    assert agent.data_parallel and isinstance(agent.training_tensors(), DataParallelState)
    with pytest.raises(ValueError):
        S.OverlappedActorLearner(agent, env)
    env.close(); mem.close()


# ---- two ranks ----------------------------------------------------------------------------------------------------
_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
import sac_agent_b200 as S
from sac_agent_b200.continuous_agent import ContinuousAgent
rank, local_rank, world = S.sharding.dist_info()
torch.cuda.set_device(local_rank)
backend, mode, out_dir = sys.argv[1], sys.argv[2], sys.argv[3]
dist.init_process_group(backend, init_method="file://" + out_dir + "/store", rank=rank, world_size=world)
kw = dict(fp32_eager=dict(learner_precision="fp32", use_cuda_graph=False),
          fp32_graph=dict(learner_precision="fp32", use_cuda_graph=True),
          tcgen05=dict(learner_precision="tcgen05"))[mode]
cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
mem = S.ReplayBuffer(100_000, (11,), 1, precision="fp32", device=local_rank, seed=20 + rank, as_torch=True)
uneven = S.BatchedBoatEnv(cfg, 1000 + rank, seed=3, precision="fp32", device=local_rank, auto_reset=True)
try:
    ContinuousAgent(cfg, None, (11,), uneven, device=local_rank, memory=mem, data_parallel=True, **kw)
    raise SystemExit("uneven shards were accepted")
except ValueError:
    pass
uneven.close()
env = S.make_sharded_env(cfg, 2048, seed=3, precision="fp32", auto_reset=True)
torch.manual_seed(100 + rank)             # different initial weights: the broadcast makes them rank 0's
agent = ContinuousAgent(cfg, None, (11,), env, device=local_rank, seed=20 + rank, memory=mem,
                        policy_precision="tcgen05", data_parallel=True, **kw)
rec = dict(initial=[t.cpu().clone() for t in agent.training_tensors()], batches=[], eps=[], losses=[])
env.reset()
for _ in range(10):
    agent.collect(env, 1)
    out = agent.learn()
    if out is not None:
        rec["batches"].append([t.cpu().clone() for t in agent._batch])
        rec["eps"].append(agent._eps.cpu().clone())
        rec["losses"].append(torch.stack([x.clone() for x in out]).cpu())
torch.cuda.synchronize()
rec["final"] = [t.cpu().clone() for t in agent.training_tensors()]
torch.save(rec, os.path.join(out_dir, f"rank{{rank}}.pt"))
dist.barrier()
env.close(); mem.close()
dist.destroy_process_group()
print("DP_OK")
"""


def _two_ranks(tmp_path, backend, mode):
    script = tmp_path / "dp_worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r if backend == "nccl" else 0))
        procs.append(subprocess.Popen([sys.executable, str(script), backend, mode, str(tmp_path)], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    for p in procs:
        out, err = p.communicate(timeout=600)
        assert p.returncode == 0 and "DP_OK" in out, err[-3000:]
    return [torch.load(tmp_path / f"rank{r}.pt") for r in range(2)]


def _emulate(mode, rec0, rec1):
    """One process: from rank 0's initial state, each update is DeviceAdam on 0.5 g0 + 0.5 g1, where g_r are the
    gradients of rank r's recorded batch and eps (the same kernels: autograd for fp32, boatagent_sac_gradients for
    tcgen05).  Returns (mean losses per update, final training tensors)."""
    prec = "tcgen05" if mode == "tcgen05" else "fp32"
    mem = S.ReplayBuffer(4096, (11,), 1, precision="fp32", device=0, as_torch=True)
    agent = ContinuousAgent(S.load_config(base_settings__experiment=6, agent__batch_size=256), None, (11,),
                            _env_stub(), device=0, memory=mem, learner_precision=prec)
    with torch.no_grad():
        for t, v in zip(agent.training_tensors(), rec0["initial"]):
            t.copy_(v)
    L, o = agent.learner, agent.learner.optimizer
    losses = []
    for it in range(len(rec0["batches"])):
        per_rank = []
        for rec in (rec0, rec1):
            for t, v in zip(agent._batch, rec["batches"][it]):
                t.copy_(v)
            agent._eps.copy_(rec["eps"][it])
            g = [torch.zeros_like(p) for p in o.params]
            lv = torch.zeros(3, device="cuda")
            if prec == "tcgen05":
                for k, x in enumerate(g):
                    o._slots[k].grad = x.data_ptr()
                assert _sac_gradients(agent, 1.0, lv) == 0
            else:
                s, a, r, s2, d = agent._batch
                L.gradients(s, a, r, s2, d.bool(), agent._eps[0], agent._eps[1], g + [lv[0], lv[1], lv[2]])
            per_rank.append((g, lv))
        (g0, l0), (g1, l1) = per_rank
        o.step([0.5 * a + 0.5 * b for a, b in zip(g0, g1)])
        losses.append(0.5 * l0 + 0.5 * l1)
    torch.cuda.synchronize()
    out = [l.cpu() for l in losses], [t.cpu().clone() for t in agent.training_tensors()]
    mem.close()
    return out


def _check_two_ranks(recs, mode):
    rec0, rec1 = recs
    assert len(rec0["batches"]) == len(rec1["batches"]) >= 9
    # the ranks sampled their own rings (the first batches can coincide: every env starts from the same observation)
    assert any(not torch.equal(a, b) for x, y in zip(rec0["batches"], rec1["batches"]) for a, b in zip(x, y))
    for a, b in zip(rec0["initial"], rec1["initial"]):
        assert torch.equal(a, b)
    for a, b in zip(rec0["final"], rec1["final"]):       # weights, target, Adam moments, step counter
        assert torch.equal(a, b)
    assert int(rec0["final"][32][0]) == len(rec0["batches"])   # DeviceAdam's step counter follows the 32 parameters
    for a, b in zip(rec0["losses"], rec1["losses"]):
        assert torch.equal(a, b)
    losses, final = _emulate(mode, rec0, rec1)
    for a, b in zip(rec0["losses"], losses):
        assert torch.equal(a, b)
    for a, b in zip(rec0["final"], final):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32_eager", "fp32_graph", "tcgen05"])
def test_two_ranks_share_one_gpu_over_gloo(mode, tmp_path):
    _check_two_ranks(_two_ranks(tmp_path, "gloo", mode), mode)


@pytest.mark.gpu
@TWO_GPUS
@pytest.mark.parametrize("mode", ["fp32_graph", "tcgen05"])
def test_two_ranks_over_nccl(mode, tmp_path):
    _check_two_ranks(_two_ranks(tmp_path, "nccl", mode), mode)


# ---- the driver -----------------------------------------------------------------------------------------------------
DRIVER_CASES = {"fp32-record": ["--record-envs", "2", "--log-every", "10"],
                "tcgen05-collect": ["--learner-precision", "tcgen05", "--policy-precision", "tcgen05",
                                    "--collect-steps", "2", "--log-every", "10"]}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(DRIVER_CASES))
def test_driver_world_1_is_the_plain_run(case, tmp_path, monkeypatch):
    import train_sac
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    common = ["--envs", "2048", "--iters", "30", "--warmup-iters", "5", "--buffer", "100000", "--experiment", "6",
              "--set", "agent__batch_size=256"] + DRIVER_CASES[case]
    plain = train_sac.main(common + ["--experiments-root", str(tmp_path / "plain")])
    dp = train_sac.main(common + ["--experiments-root", str(tmp_path / "dp"), "--data-parallel"])
    assert dp["data_parallel"] is True and dp["effective_batch"] == 256 and "data_parallel" not in plain
    for k in ("losses_v_pi_q", "episodes", "reached_goal"):
        assert dp[k] == plain[k], k
    # the return sums are fp64 atomics: equal up to the order in which episodes ended
    assert dp["mean_return"] == pytest.approx(plain["mean_return"], rel=1e-12)
    assert dp["best_interval_return"] == pytest.approx(plain["best_interval_return"], rel=1e-12, nan_ok=True)
    if "--record-envs" in DRIVER_CASES[case]:
        assert dp["recorded_envs"] == plain["recorded_envs"] == 2
    rows = [open(os.path.join(s["experiment_dir"], "console.csv")).read().count("\n") for s in (plain, dp)]
    assert rows[0] == rows[1] > 1


@pytest.mark.gpu
@TWO_GPUS
def test_driver_two_ranks_under_torchrun(tmp_path):
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "examples", "train_sac.py"), "--data-parallel", "--envs", "4096", "--iters",
                        "20", "--warmup-iters", "5", "--buffer", "100000", "--set", "agent__batch_size=256",
                        "--experiments-root", str(tmp_path), "--log-every", "10"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    assert summary["data_parallel"] is True and summary["effective_batch"] == 512 and summary["n_gpus"] == 2
    assert os.listdir(os.path.join(tmp_path, "setting_5")) == ["experiment_r0"]
