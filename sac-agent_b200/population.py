"""Population-based training across GPUs (SURVEY.md 8f rank 3).

The reference's ``main.py -p N`` (main.py:215-235) starts N independent processes, each training one model with its
own random draw of the four agent hyper-parameters (utils/hyperparameter_tuner.py:9-52: alpha, beta, gamma, tau
within the ranges of configs/hp_configs.yaml) and keeps the best score of each in overview.csv -- random search,
the members never talk.  With one member per GPU under ``torchrun`` the members can: every ``M`` iterations

  exploit   the members in the bottom quarter of the ranking (by the mean return of the episodes that ended since
            the last round) adopt the weights, optimiser state and hyper-parameters of the best member
            (one NCCL broadcast of ~4 MB per round; nothing else crosses NVLink), and
  explore   perturb the adopted hyper-parameters by x0.8 or x1.25, clipped to the tuner's ranges.

``exploit_explore`` works on any list of tensors and any process group (NCCL on GPUs, gloo in the CPU test).

On ONE GPU, ``AgentPopulation`` trains P members in one process: each member is an ordinary ``ContinuousAgent`` with its
own env, ring, experiment directory and hyper-parameters, and one ``learn()`` updates all of them in four launches (one
sample-gather for every ring, one Gaussian draw, the two kernels of the members' ``FusedLearner``).
``exploit_explore_local`` is ``exploit_explore`` over such members, with device copies instead of collectives.
With ``data_parallel``, every member is ONE agent trained by all ranks of a process group: each rank holds its own
env shard and ring of every member, and one update round of all members is one gradient launch pair, one all-reduce
and one Adam launch.
"""
from __future__ import annotations

import ctypes as C
import math
import random

from .experiment import HP_RANGES

HP_KEYS = ("alpha", "beta", "gamma", "tau")


def perturb(hp: dict, rng: random.Random, factors=(0.8, 1.25)) -> dict:
    """Explore: every hyper-parameter times a factor drawn from ``factors``, clipped to the tuner's range
    (hp_configs.yaml), rounded to 4 decimals like hyperparameter_tuner.py:24-45.  gamma is perturbed through
    1 - gamma (the effective horizon)."""
    out = {}
    for k in HP_KEYS:
        lo, hi = HP_RANGES[k]
        f = rng.choice(factors)
        v = 1.0 - (1.0 - hp[k]) * f if k == "gamma" else hp[k] * f
        out[k] = round(min(max(v, lo), hi), 4)
    return out


def select(scores, bottom_fraction: float = 0.25):
    """The ranking of one population round.  ``scores``: one per member, higher is better, NaN / -inf = no finished
    episode.  Returns (ranking best first with ties broken by index, the best member, the losers that adopt it: the
    bottom ``bottom_fraction`` (at least one) of the ranking, without the best and without members scoring as well
    as it; nobody adopts when no member has a score)."""
    n = len(scores)
    ranking = sorted(range(n), key=lambda r: (-scores[r], r))
    best = ranking[0]
    n_bottom = max(1, int(n * bottom_fraction)) if scores[best] > -float("inf") else 0
    return ranking, best, [r for r in ranking[n - n_bottom:] if r != best and scores[r] < scores[best]]


def exploit_explore(tensors, hp: dict, score: float, rng: random.Random, bottom_fraction: float = 0.25, group=None):
    """One population round.  ``tensors``: this member's state (parameters, optimiser moments, ...) as a list of
    tensors with the same shapes on every member; ``hp``: its hyper-parameters (HP_KEYS); ``score``: higher is better
    (NaN = no finished episode: ranks last).  Returns (hp, info): the hyper-parameters to continue with, and a dict
    {"adopted_from": rank or None, "ranking": [...], "scores": [...]}.  Tensors are overwritten in place when this
    member adopts.  Collective: every member of ``group`` must call it."""
    import torch
    import torch.distributed as dist
    from .continuous_agent import DataParallelState
    if isinstance(tensors, DataParallelState):
        raise ValueError("exploit_explore: these are the tensors of a data-parallel agent, one agent shared by its "
                         "ranks; population rounds need one agent per member")
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) < 2:
        return dict(hp), {"adopted_from": None, "ranking": [0], "scores": [score]}
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = tensors[0].device
    mine = torch.tensor([score if not math.isnan(score) else -float("inf")] + [float(hp[k]) for k in HP_KEYS],
                        dtype=torch.float64, device=dev)
    table = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(table, mine, group=group)
    table = torch.stack(table).cpu()
    scores = table[:, 0].tolist()
    ranking, best, losers = select(scores, bottom_fraction)              # ties by rank: the same everywhere
    info = {"adopted_from": None, "ranking": ranking, "scores": scores}
    if not losers:
        return dict(hp), info
    # one flat broadcast of the best member's state; only the losers keep it
    flat = torch.cat([t.detach().reshape(-1).to(torch.float32) if t.is_floating_point() else t.detach().reshape(-1).double().float()
                      for t in tensors]) if rank == best else \
        torch.empty(sum(t.numel() for t in tensors), dtype=torch.float32, device=dev)
    src = dist.get_global_rank(group, best) if group is not None else best
    dist.broadcast(flat, src=src, group=group)
    if rank not in losers:
        return dict(hp), info
    off = 0
    with torch.no_grad():
        for t in tensors:
            n = t.numel()
            t.copy_(flat[off:off + n].reshape(t.shape).to(t.dtype))
            off += n
    info["adopted_from"] = best
    best_hp = dict(zip(HP_KEYS, table[best, 1:].tolist()))
    return perturb(best_hp, rng), info


def exploit_explore_local(members, scores, rng: random.Random, bottom_fraction: float = 0.25):
    """``exploit_explore`` for members held by one process (``ContinuousAgent`` objects on one device): the same
    ranking (``select``) and perturbation, with each loser's ``training_tensors()`` overwritten by device copies of the
    best member's.  ``scores``: one per member (NaN = no finished episode).  Returns
    {"ranking", "scores", "best", "adopted": {loser index: perturbed hyper-parameters}}."""
    import torch
    scores = [-float("inf") if math.isnan(float(x)) else float(x) for x in scores]
    if len(scores) != len(members):
        raise ValueError(f"exploit_explore_local: {len(scores)} scores for {len(members)} members")
    ranking, best, losers = select(scores, bottom_fraction)
    info = {"ranking": ranking, "scores": scores, "best": best, "adopted": {}}
    if not losers:
        return info
    src, best_hp = members[best].training_tensors(), members[best].hyperparameters()
    for r in losers:
        with torch.no_grad():
            torch._foreach_copy_(members[r].training_tensors(), src)
        hp = perturb(best_hp, rng)
        members[r].set_hyperparameters(**hp)
        members[r]._weights_changed()
        info["adopted"][r] = hp
    return info


class AgentPopulation:
    """P independent SAC members on one GPU, updated together (the reference's ``main.py -p P`` on one device).

    Member m of process ``rank`` has the global index g = rank * P + m.  It is a ``ContinuousAgent`` with
    policy and learner precision "tcgen05", its own ``BatchedBoatEnv`` (``envs_per_member`` envs, global env ids from
    g * envs_per_member, so no two members share wind draws), its own ``ReplayBuffer`` (ring seed ``seed + g``), its
    initial weights drawn under torch seed ``seed + g`` and its tcgen05 acting seed 0x5ac + g.  With P = 1 and rank 0
    that is the agent ``examples/train_sac.py`` builds with the same seed, bit for bit.

    ``data_parallel``: a torch.distributed process group (True: the default group) of W ranks that train every member
    together; ``rank`` is then the rank r in that group.  Each rank holds ``envs_per_member`` envs of each member
    (global env ids from (m W + r) envs_per_member, so a member's W shards are contiguous), its own ring of each member
    (ring seed ``seed + r P + m``) and its own acting seed 0x5ac + r P + m.  The initial weights are drawn under torch
    seed ``seed + m`` and rank 0's training tensors are broadcast once; every rank must pass the same P, batch size and
    ``envs_per_member`` (checked here).  ``learn()`` computes every member's gradients of this rank's batch times 1 / W,
    sums them over the ranks with one all-reduce and applies the same Adam step on every rank, so the members stay
    bit-identical across ranks (1 / W is exact for power-of-two W).  At W = 1 this is the plain population, bit for
    bit.  Population rounds (``exploit_explore``) keep the ranks identical when every rank passes the same scores
    (``counters()`` sums them over the ranks) and an identically seeded rng.

    ``configs``: one config per member (e.g. its tuned_configs.yaml draw), else ``config`` for all; the batch size must
    be the same.  Change a member's hyper-parameters through ``set_hyperparameters`` or ``exploit_explore`` so that
    the next ``learn()`` sees them.

    ``algorithm``: "sac1" or "sac2" (``ContinuousAgent(algorithm=...)``; every member's SAC-v2 update runs in the same
    launches).  ``target_entropy``, ``init_temperature`` and ``temperature_lr`` (sac2 only): one value for every member
    or a sequence of one per member.  SAC-v2 does not train data-parallel."""

    def __init__(self, config, members, envs_per_member, seed=0, rank=0, device=None, configs=None,
                 experiment_dirs=None, buffer_size=None, done_flag_mode=1, data_parallel=None, algorithm="sac1",
                 target_entropy=None, init_temperature=1.0, temperature_lr=None):
        import torch
        from . import _lib
        from .boat_env import BatchedBoatEnv
        from .buffer import ReplayBuffer
        from .continuous_agent import ContinuousAgent, FusedLearner
        from .networks import TensorCorePolicy
        P = int(members)
        if not 1 <= P <= 16:
            raise ValueError(f"AgentPopulation: 1 to 16 members per process (BOATAGENT_SAC_MAX_MEMBERS), got {P}")
        if algorithm not in ("sac1", "sac2"):
            raise ValueError(f"AgentPopulation: algorithm sac1 or sac2, got {algorithm!r}")
        if algorithm == "sac2" and data_parallel is not None and data_parallel is not False:
            raise ValueError("AgentPopulation: algorithm='sac2' does not train data-parallel")
        if algorithm == "sac1" and (target_entropy is not None or init_temperature != 1.0 or temperature_lr is not None):
            raise ValueError("AgentPopulation: target_entropy, init_temperature and temperature_lr belong to "
                             "algorithm='sac2'")

        def per_member(x, name):
            xs = list(x) if isinstance(x, (list, tuple)) else [x] * P
            if len(xs) != P:
                raise ValueError(f"AgentPopulation: {name} needs one value or one per member ({P})")
            return xs
        v2 = [{} for _ in range(P)]
        if algorithm == "sac2":
            for name, x in (("target_entropy", target_entropy), ("init_temperature", init_temperature),
                            ("temperature_lr", temperature_lr)):
                for m, v in enumerate(per_member(x, name)):
                    v2[m][name] = v
        configs = list(configs) if configs is not None else [config] * P
        dirs = list(experiment_dirs) if experiment_dirs is not None else [None] * P
        if len(configs) != P or len(dirs) != P:
            raise ValueError("AgentPopulation: one config and one experiment directory per member")
        self.batch_size = int(configs[0].agent.batch_size)
        if any(int(c.agent.batch_size) != self.batch_size for c in configs):
            raise ValueError("AgentPopulation: the members share one batch size")
        self._L, self._lib = _lib.lib(), _lib
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self._dp = None   # (group, world) in data-parallel mode
        if data_parallel is not None and data_parallel is not False:
            import torch.distributed as dist
            if not (dist.is_available() and dist.is_initialized()):
                raise ValueError("AgentPopulation: data_parallel needs an initialised torch.distributed process group")
            group = None if data_parallel is True else data_parallel
            self._dp = (group, dist.get_world_size(group))
            rank = dist.get_rank(group)
        self.rank, self.seed, self.done_flag_mode = int(rank), int(seed), int(done_flag_mode)
        W, E = (self._dp[1] if self._dp else 1), int(envs_per_member)
        self.envs, self.members = [], []
        for m in range(P):
            g = self.rank * P + m
            cfg = configs[m]
            # data-parallel: member m's W shards are contiguous, and its weights do not depend on the rank
            first_env, weight_seed = ((m * W + self.rank) * E, seed + m) if self._dp else (g * E, seed + g)
            env = BatchedBoatEnv(cfg, E, seed=seed, precision="fp32", device=self.device.index,
                                 env_id_offset=first_env, auto_reset=True)
            size = int(cfg.agent.max_size) if buffer_size is None else int(buffer_size)
            mem = ReplayBuffer(size, (11,), 1, precision="fp32", device=self.device.index, seed=seed + g, as_torch=True)
            with torch.random.fork_rng(devices=[self.device]):
                torch.manual_seed(weight_seed)
                agent = ContinuousAgent(cfg, dirs[m], env.observation_space.shape, env, device=self.device.index,
                                        seed=seed + g, memory=mem, policy_precision="tcgen05",
                                        learner_precision="tcgen05", algorithm=algorithm, **v2[m])
            agent._tc_policy = TensorCorePolicy(agent.actor, seed=0x5ac + g)
            self.envs.append(env)
            self.members.append(agent)
        B = self.batch_size
        # the members' Gaussian draws are slices of one tensor: one normal_() per learn()
        self.eps = torch.zeros((P, 2, B, 1), dtype=torch.float32, device=self.device)
        self._sample = (_lib.SampleMember * P)()
        for m, a in enumerate(self.members):
            a._eps = self.eps[m]
            s, act, r, s2, d = a._batch
            self._sample[m] = _lib.SampleMember(a.memory._h, 0, 0, s.data_ptr(), act.data_ptr(), r.data_ptr(),
                                                s2.data_ptr(), d.data_ptr())
        self._flat = None
        if self._dp is not None:
            self._init_data_parallel(E)
        self._learner = FusedLearner(self.members)

    def _init_data_parallel(self, envs_per_member):
        """Checks that every rank holds the same population, points every member's gradients and losses into one flat
        [P, n_params + 3] buffer (one all-reduce per round) and starts every rank from rank 0's members."""
        import torch
        import torch.distributed as dist
        from .continuous_agent import point_grads_into
        group, world = self._dp
        P = len(self.members)
        shape = torch.tensor([P, self.batch_size, envs_per_member], dtype=torch.int64, device=self.device)
        both = torch.cat([shape, -shape])
        dist.all_reduce(both, op=dist.ReduceOp.MAX, group=group)
        if not torch.equal(both[:3], -both[3:]):
            raise ValueError(f"AgentPopulation: every rank of the data-parallel group needs the same members, batch "
                             f"size and envs per member (this rank: {P}, {self.batch_size}, {envs_per_member}; "
                             f"largest over the ranks: {both[:3].tolist()})")
        n = sum(p.numel() for p in self.members[0].learner.optimizer.params)
        self._flat = torch.zeros((P, n + 3), dtype=torch.float32, device=self.device)
        for m, a in enumerate(self.members):
            point_grads_into(a, self._flat[m])
        src = 0 if group is None else dist.get_global_rank(group, 0)
        for a in self.members:
            for t in a.training_tensors():
                dist.broadcast(t, src=src, group=group)
            a._weights_changed()

    @property
    def data_parallel(self):
        """True when every member is trained by a process group (constructor argument ``data_parallel``)."""
        return self._dp is not None

    def __len__(self):
        return len(self.members)

    def reset(self):
        """Resets every member's env; returns their observations."""
        return [env.reset() for env in self.envs]

    def collect(self, steps):
        """``steps`` env steps of every member's envs (``ContinuousAgent.collect``, one launch per member).  Each
        member's packed acting weights are refreshed once, here, instead of after every update."""
        for a, env in zip(self.members, self.envs):
            a._tc_policy.refresh()
            a.collect(env, steps, done_flag_mode=self.done_flag_mode)

    def learn(self):
        """One update of every member: the batched sample-gather, one Gaussian draw for all, and the two kernels of
        the members' fused update (``FusedLearner.update``, no sync; SAC-v2: three kernels).  Returns each member's
        (value, actor, critic) losses -- SAC-v2: (temperature, actor, critic) -- as device tensors, or None (nothing launched) while some member's ring holds less than a batch.

        Data-parallel: the update is ``FusedLearner.gradients`` (times 1 / W), one all-reduce (SUM) of every member's
        gradients and losses, and ``FusedLearner.adam``; the losses are the means over the ranks.  The rank shards are
        equal, so all ranks start updating at the same call without a vote."""
        if any(a.memory.mem_cntr < self.batch_size for a in self.members):
            return None
        import torch
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        for m, a in enumerate(self.members):   # load_state_dict may have changed the seed
            self._sample[m].seed, self._sample[m].counter = a.memory.seed, a.memory._samples
        self._lib.check(self._L.boatreplay_sample_members(self._sample, len(self.members), self.batch_size, stream),
                        "boatreplay_sample_members")
        for a in self.members:
            a.memory._samples += 1
        self.eps.normal_()
        if self._dp is None:
            self._learner.update()
        else:
            import torch.distributed as dist
            group, world = self._dp
            self._learner.gradients(1.0 / world)
            dist.all_reduce(self._flat, op=dist.ReduceOp.SUM, group=group)
            self._learner.adam()
        for a in self.members:
            a.updates += 1
        return [a._losses for a in self.members]

    def counters(self):
        """Each member's episode counters (``BatchedBoatEnv.counters()`` dicts), in member order.  Data-parallel: summed
        over the ranks with one all-reduce of a [P, 8] float64 tensor (collective), so every rank gets the same."""
        if self._dp is None:
            return [env.counters() for env in self.envs]
        import torch
        import torch.distributed as dist
        from .boat_env import COUNTER_NAMES
        c = torch.stack([env.counters_tensor() for env in self.envs])
        dist.all_reduce(c, op=dist.ReduceOp.SUM, group=self._dp[0])
        return [dict(zip(COUNTER_NAMES, row)) for row in c.cpu().tolist()]

    def set_hyperparameters(self, m, **hp):
        """``ContinuousAgent.set_hyperparameters`` of member m, seen by the next ``learn()``."""
        self.members[m].set_hyperparameters(**hp)

    def exploit_explore(self, scores, rng: random.Random, bottom_fraction: float = 0.25):
        """One population round over the members (``exploit_explore_local``).  Data-parallel: every rank must call it
        with the same scores (e.g. from ``counters()``) and an identically seeded rng, so that all ranks make the same
        round and their members stay bit-identical."""
        return exploit_explore_local(self.members, scores, rng, bottom_fraction)

    def state_dict(self):
        """The members' ``ContinuousAgent.state_dict()``, in member order."""
        return [a.state_dict() for a in self.members]

    def load_state_dict(self, sd):
        if len(sd) != len(self.members):
            raise ValueError(f"checkpoint of {len(sd)} members for a population of {len(self.members)}")
        for a, s in zip(self.members, sd):
            a.load_state_dict(s)

    def close(self):
        for a, env in zip(self.members, self.envs):
            env.close()
            a.memory.close()
