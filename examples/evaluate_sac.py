#!/usr/bin/env python
"""Evaluate a trained actor over many envs: the reference's `main.py -r` (render_model, main.py:137-172, without
the rendering), batched.  The actor saved by `train_sac.py --experiments-root` is loaded with `load_models` and
every env runs one fresh episode per round under it, the policy and the env step fused in one kernel per round
(TensorCorePolicy.rollout, csrc/rollout.cu; the policy acts with bf16 inputs and fp32 accumulation).

    python examples/evaluate_sac.py --checkpoints experiments/setting_6/experiment_r0_... --envs 65536
    python examples/evaluate_sac.py --checkpoints DIR --rounds 4 --stochastic --record-envs 4
    torchrun --nproc-per-node 8 examples/evaluate_sac.py --checkpoints DIR --envs 1048576

`--record-envs K` writes the reference's Recorder CSVs (episodes/) of the first K envs of round 1 (of rank 0's
shard) under --output.  They are replayed through the per-step path (TensorCorePolicy.act, BatchedBoatEnv.step,
DeviceRecorder) with the same seeds: env draws are keyed by global env id and policy draws by (seed; row, step), so
these are the same episodes.  The policy's seed is --seed and the rank, so shards draw independent noise.
Multi-GPU: each rank evaluates its shard, the summary counters are all-reduced.  The last line printed is a JSON
summary.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200.csv_export import INFO_COLUMNS, EpisodeBook, _append_rows  # noqa: E402
from sac_agent_b200.networks import TensorCorePolicy  # noqa: E402


def record_first_envs(agent, env, k, step0, max_steps, steps_taken, deterministic, out_dir):
    """Replays env rows 0 .. k-1 of `env`'s round (started with policy step `step0`) through the per-step path and
    records each env up to the end of its episode (`steps_taken` [k] from the rollout).  As in main.py:79-81, a data
    row is the state BEFORE a step: the reset state, then the state after every step but the last, so the terminal
    state is never written; the last step of an ended episode only adds its info.csv row."""
    renv = S.BatchedBoatEnv(env.config, k, seed=env.seed, precision="fp32", device=env.device.index,
                            env_id_offset=env.env_id_offset, auto_reset=False)
    pol = TensorCorePolicy(agent.actor, seed=agent.tensor_core_policy().seed)
    pol.steps = step0
    ids = list(range(env.env_id_offset, env.env_id_offset + k))
    book = EpisodeBook(ids, out_dir)   # one naming for all k envs (env<id>_...)
    renv.reset()
    recs = []
    for i in ids:   # one recorder per env: each stops at the end of its own episode
        rec = S.DeviceRecorder(renv, [i], out_dir, capacity=1024)
        rec.book = book
        rec.start()
        recs.append(rec)
    eps = torch.zeros((k, 1), dtype=torch.float32, device=renv.device) if deterministic else None
    for t in range(min(max_steps, max(steps_taken))):
        a = pol.act(renv.obs, eps=eps).reshape(-1)
        renv.step(a)
        for j, (i, rec) in enumerate(zip(ids, recs)):
            if t + 1 < steps_taken[j] or (t + 1 == steps_taken[j] and not int(renv.term[j])):
                rec.capture(a)
            elif t + 1 == steps_taken[j]:   # the episode ended on this step: its info.csv row, no data row
                rec.close()
                vals = [np.float64(x) for x in (a[j].item(), renv.reward[j].item())]
                path, row = book.after_step(i, vals[0], vals[1], int(renv.term[j]))
                _append_rows(path, INFO_COLUMNS, [row])
    for rec in recs:
        rec.close()
    renv.close()


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--checkpoints", required=True, help="experiment directory written by train_sac.py "
                                                          "--experiments-root (its checkpoints/ is loaded)")
    ap.add_argument("--envs", type=int, default=65536, help="total envs over all ranks")
    ap.add_argument("--experiment", type=int, default=6)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--max-steps", type=int, default=None,
                    help="steps per round (default: enough for every episode to end, at the latest by timeout)")
    ap.add_argument("--stochastic", action="store_true", help="draw actions as in training (default: tanh(mean))")
    ap.add_argument("--rounds", type=int, default=1, help="reset() + rollout R times: R fresh episodes per env")
    ap.add_argument("--record-envs", type=int, default=0, metavar="K",
                    help="write the Recorder CSVs (episodes/) of the first K envs of round 1 (rank 0)")
    ap.add_argument("--output", default=None, help="directory of the recorded episodes/ (default: "
                                                   "<checkpoints>/evaluation)")
    args = ap.parse_args(argv)
    if args.rounds < 1 or args.envs < 1:
        ap.error("--rounds and --envs must be positive")

    rank, local_rank, world = S.sharding.dist_info()
    torch.cuda.set_device(local_rank)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = S.load_config(base_settings__experiment=args.experiment)
    env = S.make_sharded_env(cfg, args.envs, seed=args.seed, precision="fp32", auto_reset=False)
    mem = S.ReplayBuffer(int(cfg.agent.batch_size), (11,), 1, precision="fp32", device=local_rank, seed=args.seed,
                         as_torch=True)   # the agent needs one; evaluation stores nothing
    # a SAC-v2 directory (train_sac.py --algorithm sac2) holds target critics instead of value networks
    sac2 = os.path.exists(os.path.join(args.checkpoints, "checkpoints", "target_critic_network_1"))
    agent = S.ContinuousAgent(cfg, args.checkpoints, env.observation_space.shape, env, device=local_rank,
                              seed=args.seed + rank, memory=mem, algorithm="sac2" if sac2 else "sac1")
    agent.load_models()
    # policy draws are keyed by (seed; row, step) and rows restart at 0 on every shard: a seed per rank keeps the
    # shards' noise independent under --stochastic
    agent.tensor_core_policy().seed = (args.seed << 16) + rank
    deterministic = not args.stochastic
    max_steps = args.max_steps or int(math.ceil(env.params.t_max / env.params.dt)) + 1
    n_kinds = len(S.TERM_NAMES) - 1
    # summed over rounds and ranks: [counts per kind, episodes, running, return sum, return sum of squares, length sum]
    tot = torch.zeros(n_kinds + 5, dtype=torch.float64, device=env.device)
    lo_hi = torch.tensor([math.inf, math.inf], dtype=torch.float64, device=env.device)   # [min, -max] return
    recorded = None
    for rnd in range(args.rounds):
        env.reset()
        step0 = agent.tensor_core_policy().steps
        ret, steps, term, _ = agent.evaluate(env, max_steps, deterministic)
        ended = term != 0
        r = ret.double()[ended]
        for k in range(n_kinds):
            tot[k] += (term == k + 1).sum()
        tot[n_kinds] += ended.sum()
        tot[n_kinds + 1] += (~ended).sum()
        tot[n_kinds + 2] += r.sum()
        tot[n_kinds + 3] += (r * r).sum()
        tot[n_kinds + 4] += steps[ended].double().sum()
        if r.numel():
            lo_hi = torch.minimum(lo_hi, torch.stack([r.min(), -r.max()]))
        if rnd == 0 and args.record_envs and rank == 0:
            k = min(args.record_envs, env.n_envs)
            taken = steps[:k].tolist()
            out = args.output or os.path.join(args.checkpoints, "evaluation")
            record_first_envs(agent, env, k, step0, max_steps, taken, deterministic, out)
            recorded = {"recorded_envs": k, "recorded_steps": taken, "recorded_term": term[:k].tolist(),
                        "recorded_dir": out}
    if world > 1:
        torch.distributed.all_reduce(tot)
        torch.distributed.all_reduce(lo_hi, op=torch.distributed.ReduceOp.MIN)
    tot, lo_hi = tot.tolist(), lo_hi.tolist()
    episodes = tot[n_kinds]
    mean = tot[n_kinds + 2] / episodes if episodes else float("nan")
    summary = {"example": "evaluate_sac", "checkpoints": args.checkpoints, "n_gpus": world, "envs": args.envs,
               "rounds": args.rounds, "max_steps": max_steps, "deterministic": deterministic,
               "episodes": int(episodes), "running": int(tot[n_kinds + 1]),
               "terminations": {S.TERM_NAMES[k + 1]: int(tot[k]) for k in range(n_kinds)},
               "goal_fraction": tot[0] / (args.envs * args.rounds),
               "return_mean": mean,
               "return_std": math.sqrt(max(tot[n_kinds + 3] / episodes - mean * mean, 0.0)) if episodes else float("nan"),
               "return_min": lo_hi[0] if episodes else float("nan"),
               "return_max": -lo_hi[1] if episodes else float("nan"),
               "length_mean": tot[n_kinds + 4] / episodes if episodes else float("nan")}
    if recorded:
        summary.update(recorded)
    if rank == 0:
        print(json.dumps(summary), flush=True)
    env.close()
    mem.close()
    if world > 1:
        torch.distributed.destroy_process_group()
    return summary


if __name__ == "__main__":
    main()
