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
"""
from __future__ import annotations

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
    ranking = sorted(range(world), key=lambda r: (-scores[r], r))       # best first; ties by rank: the same everywhere
    best = ranking[0]
    n_bottom = max(1, int(world * bottom_fraction)) if scores[best] > -float("inf") else 0
    losers = [r for r in ranking[world - n_bottom:] if r != best and scores[r] < scores[best]]
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
