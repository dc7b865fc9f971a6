#!/usr/bin/env python
"""End-to-end SAC (v1: actor, twin critics, value + target value) on the GPU-resident batched BoatEnv
and the fused device replay buffer -- BASELINE.json configs[4] / SURVEY.md 8(f) rank 1.  `--algorithm sac2` trains
SAC with twin target critics and a learned entropy temperature instead (SAC2Learner); its JSON summary adds
`algorithm` and the final `temperature`.  `--prioritized` draws the updates' batches by prioritized experience replay
(ContinuousAgent(prioritized=True)); its JSON summary adds `prioritized` and the four priority parameters.

The loop is the reference's main.py:72-90 with every piece on the device:

    action = agent.choose_action(obs)            -> ContinuousAgent.choose_action_graphed (N envs, one graph)
    obs_, r, done, info = env.step(action)       \\  ContinuousAgent.step_and_remember: ONE kernel
    agent.remember(obs, action, r, obs_, done)   /   (boatenv_step_store)
    agent.learn()                                -> sample-gather kernel + one captured CUDA graph

Algorithm and hyper-parameters are the reference's (agent/continuous_agent.py:96-154,
networks/networks.py, the `agent:` block of original_config.yaml); the update is checked against a
recorded run of the reference's own learn() in tests/test_agent_golden.py.

    python examples/train_sac.py --envs 65536 --iters 200
    python examples/train_sac.py --envs 8192 --policy-precision tcgen05 --collect-steps 8 --updates-per-iter 8
                                          # 8 steps of act + step + remember per launch (ContinuousAgent.collect)
    torchrun --nproc-per-node 8 examples/train_sac.py --envs 65536        # replicas: one agent per GPU shard
    torchrun --nproc-per-node 8 examples/train_sac.py --experiments-root experiments --tune
                                          # the reference's `main.py -p 8`: a tuned_configs.yaml draw per member
    torchrun --nproc-per-node 8 examples/train_sac.py --envs 65536 --data-parallel
                                          # ONE agent over all ranks: every update averages 8 batches' gradients
    python examples/train_sac.py --envs 8192 --population 8 --policy-precision tcgen05 --learner-precision tcgen05 \
        --collect-steps 8 --updates-per-iter 8 --tune    # 8 members on one GPU (AgentPopulation): one update launch pair
    torchrun --nproc-per-node 8 examples/train_sac.py --envs 65536 --population 8 --data-parallel --tune --pbt-every 50 \
        --policy-precision tcgen05 --learner-precision tcgen05 --collect-steps 8
                                          # 8 members, each ONE agent over all ranks, with population rounds

By default multi-GPU is "replicas only" (SURVEY.md 8e): every rank trains its own agent on its own env shard,
like the reference's `-p` mode runs independent models; only the episode statistics are all-reduced.
`--data-parallel` trains one agent instead: each rank samples its own ring, one all-reduce per update averages the
gradients, and rank 0 writes the one experiment directory from the all-reduced episode statistics.
The last line printed by rank 0 is a JSON summary (device-timed after `--warmup-iters`).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import sac_agent_b200 as S  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536, help="total envs over all ranks")
    ap.add_argument("--iters", type=int, default=200, help="iterations: env steps (each over every env), or "
                    "--collect-steps of them each")
    ap.add_argument("--warmup-iters", type=int, default=20, help="untimed iterations (graph capture happens here)")
    ap.add_argument("--updates-per-iter", type=int, default=1)
    ap.add_argument("--experiment", type=int, default=5)
    ap.add_argument("--buffer", type=int, default=1_000_000, help="ring capacity per rank (original_config max_size)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--log-every", type=int, default=50)
    ap.add_argument("--no-graph", action="store_true", help="eager update / policy (for comparison)")
    ap.add_argument("--experiments-root", default=None,
                    help="write the reference's experiment tree (configs/, checkpoints/, console.csv, overview.csv, "
                         "terminations.csv; main.py:116-133) under this directory, one experiment per rank")
    ap.add_argument("--tune", action="store_true",
                    help="population mode (main.py -p): every rank trains with its own tuned_configs.yaml draw")
    ap.add_argument("--policy-precision", default="fp32", choices=["fp32", "tf32", "bf16", "tcgen05"],
                    help="dense layers of choose_action on tensor-core inputs (acting only; the learner stays fp32)")
    ap.add_argument("--learner-precision", default="fp32", choices=["fp32", "tcgen05"],
                    help="tcgen05: each update runs as libboatenv's two fused kernels (bf16 operands for the 256-wide "
                         "products, fp32 accumulation) instead of the captured fp32 graph; the batch size must be a "
                         "multiple of 128")
    ap.add_argument("--set", action="append", default=[], metavar="SECTION__KEY=VALUE",
                    help="override a config key, e.g. --set agent__learning_rate_alpha=0.001 (original_config.yaml names)")
    ap.add_argument("--pbt-every", type=int, default=0,
                    help="population-based training (with torchrun, one member per GPU): every this many iterations the "
                         "bottom quarter adopts the best member's weights + hyper-parameters and perturbs them")
    ap.add_argument("--overlap", action="store_true",
                    help="acting and learning on two streams (OverlappedActorLearner: the policy lags one update)")
    ap.add_argument("--record-envs", type=int, default=0, metavar="K",
                    help="record every step of the first K envs of each rank's shard into its experiment's episodes/ "
                         "(the reference's Recorder CSVs, DeviceRecorder); flushed at every log interval")
    ap.add_argument("--collect-steps", type=int, default=0, metavar="T",
                    help="one iteration = T env steps of every env collected by ONE fused kernel (policy, env step with "
                         "auto-reset and replay store; ContinuousAgent.collect), then --updates-per-iter updates; "
                         "needs --policy-precision tcgen05.  0: one env step per iteration, policy and step launched "
                         "separately")
    ap.add_argument("--data-parallel", action="store_true",
                    help="train ONE agent over all ranks (ContinuousAgent(data_parallel=True)): every update all-reduces "
                         "the gradients of the ranks' batches, an effective batch of world x batch_size; --envs must "
                         "divide evenly over the ranks")
    ap.add_argument("--population", type=int, default=0, metavar="P",
                    help="train P independent members per process on its GPU (AgentPopulation, 1 to 16): each on the "
                         "env shard a replica gets, with its own ring, experiment directory and --tune draw; every "
                         "update round is one batched launch pair for all members.  Needs both precisions tcgen05 and "
                         "--collect-steps.  With --data-parallel under torchrun (2+ ranks) every member is ONE agent "
                         "trained by all ranks, --envs counts each member's envs over all ranks, and --tune and "
                         "--pbt-every draw and rank the members the same way on every rank")
    ap.add_argument("--algorithm", default="sac1", choices=["sac1", "sac2"],
                    help="sac1: the reference's SAC-v1 (value + target value networks, entropy weight fixed by the "
                         "reward scale); sac2: twin target critics and a learned entropy temperature (SAC2Learner)")
    ap.add_argument("--target-entropy", type=float, default=None,
                    help="sac2: the temperature's target entropy (default: minus the number of actions, -1)")
    ap.add_argument("--init-temperature", type=float, default=None, help="sac2: initial alpha (default 1.0)")
    ap.add_argument("--temperature-lr", type=float, default=None,
                    help="sac2: Adam learning rate of log alpha (default: the critics', learning_rate_beta)")
    ap.add_argument("--prioritized", action="store_true",
                    help="prioritized experience replay (Schaul et al. 2016): batches drawn by priority, critic loss "
                         "rows weighted by importance, priorities set from the TD errors")
    ap.add_argument("--priority-alpha", type=float, default=None, help="--prioritized: priority exponent (default 0.6)")
    ap.add_argument("--priority-beta", type=float, default=None,
                    help="--prioritized: initial importance-weight exponent (default 0.4)")
    ap.add_argument("--priority-beta-updates", type=int, default=None,
                    help="--prioritized: updates over which beta rises linearly to 1 (default 0: constant)")
    ap.add_argument("--priority-eps", type=float, default=None,
                    help="--prioritized: added to |TD| before the exponent (default 1e-6)")
    args = ap.parse_args(argv)
    priority_flags = (args.priority_alpha, args.priority_beta, args.priority_beta_updates, args.priority_eps)
    if not args.prioritized and any(x is not None for x in priority_flags):   # checked before any CUDA work
        ap.error("--priority-alpha, --priority-beta, --priority-beta-updates and --priority-eps need --prioritized")
    if args.prioritized:
        for flag, on in (("--data-parallel", args.data_parallel), ("--population", args.population),
                         ("--overlap", args.overlap)):
            if on:
                ap.error(f"--prioritized and {flag} cannot be combined")
        p = _priority_args(args)
        if not (p["priority_alpha"] >= 0 and 0 <= p["priority_beta"] <= 1 and p["priority_beta_updates"] >= 0
                and p["priority_eps"] > 0):
            ap.error("--priority-alpha >= 0, 0 <= --priority-beta <= 1, --priority-beta-updates >= 0 and "
                     "--priority-eps > 0")
    if args.algorithm == "sac2":   # checked before any CUDA work
        for flag, on in (("--data-parallel", args.data_parallel), ("--overlap", args.overlap)):
            if on:
                ap.error(f"--algorithm sac2 and {flag} cannot be combined")
        if args.init_temperature is not None and not args.init_temperature > 0:
            ap.error("--init-temperature must be positive")
    elif any(x is not None for x in (args.target_entropy, args.init_temperature, args.temperature_lr)):
        ap.error("--target-entropy, --init-temperature and --temperature-lr need --algorithm sac2")
    if args.record_envs and not args.experiments_root:
        ap.error("--record-envs requires --experiments-root")
    if args.collect_steps < 0:
        ap.error("--collect-steps must be >= 0")
    if args.collect_steps:   # checked before any CUDA work
        if args.policy_precision != "tcgen05":
            ap.error("--collect-steps acts through the fused tcgen05 kernel: it needs --policy-precision tcgen05")
        if args.overlap:
            ap.error("--collect-steps and --overlap cannot be combined")
        if args.record_envs:
            ap.error("--collect-steps and --record-envs cannot be combined (the fused kernel records no steps)")

    rank, local_rank, world = S.sharding.dist_info()
    if args.population:   # checked before any CUDA work
        if not 1 <= args.population <= 16:
            ap.error("--population takes 1 to 16 members per process")
        if args.policy_precision != "tcgen05" or args.learner_precision != "tcgen05":
            ap.error("--population needs --policy-precision tcgen05 and --learner-precision tcgen05")
        if args.collect_steps < 1:
            ap.error("--population needs --collect-steps T >= 1")
        for flag, on in (("--data-parallel", args.data_parallel and world < 2), ("--overlap", args.overlap),
                         ("--record-envs", args.record_envs)):
            if on:
                ap.error(f"--population and {flag} cannot be combined" +
                         (" on one process (a one-rank group is plain --population)" if flag == "--data-parallel" else ""))
        if args.pbt_every and world > 1 and not args.data_parallel:
            ap.error("--population with --pbt-every runs on one process: population rounds across ranks hold one "
                     "member per rank (or add --data-parallel: every member trained by all ranks)")
        if args.data_parallel and args.envs % world:
            ap.error(f"--population --data-parallel needs --envs (each member's envs over all ranks) divisible by the "
                     f"world size ({args.envs} envs, {world} ranks)")
        torch.cuda.set_device(local_rank)
        if world > 1:
            torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        try:
            return train_population(args, rank, local_rank, world,
                                    group=torch.distributed.group.WORLD if args.data_parallel else None)
        finally:
            if world > 1:
                torch.distributed.destroy_process_group()
    if args.prioritized and args.pbt_every and world > 1:
        ap.error("--prioritized and --pbt-every across ranks cannot be combined (population rounds between ranks hand "
                 "over weights, not the priorities of each rank's ring)")
    if args.algorithm == "sac2" and args.pbt_every and world > 1:
        ap.error("--algorithm sac2 and --pbt-every across ranks cannot be combined (population rounds between ranks "
                 "are SAC-v1's; use --population for SAC-v2 population rounds on one GPU)")
    if args.data_parallel:   # checked before any CUDA work
        for flag, on in (("--tune", args.tune), ("--pbt-every", args.pbt_every), ("--overlap", args.overlap)):
            if on:
                ap.error(f"--data-parallel and {flag} cannot be combined")
        if args.envs % world:
            ap.error(f"--data-parallel needs --envs divisible by the world size ({args.envs} envs, {world} ranks)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    elif args.data_parallel:   # a one-rank group: the agent all-reduces as it would over several
        torch.distributed.init_process_group("nccl", store=torch.distributed.HashStore(), rank=0, world_size=1,
                                             device_id=torch.device("cuda", local_rank))
    torch.manual_seed(args.seed + rank)
    overrides = {}
    for item in args.set:
        k, v = item.split("=", 1)
        overrides[k] = float(v) if any(ch in v for ch in ".e") else int(v)
    cfg = S.load_config(base_settings__experiment=args.experiment, **overrides)
    exp = None
    if args.experiments_root and not (args.data_parallel and rank > 0):   # data-parallel: rank 0's directory only   # utils/build_experiment.py: one experiment directory per population member
        import random
        exp = S.Experiment(experiment_name=f"experiment_r{rank}", subdir=f"setting_{args.experiment}",
                           root=args.experiments_root, rng=random.Random(args.seed + rank))
        tuned = exp.save_configs(cfg)
        if args.tune:
            cfg = tuned
    env = S.make_sharded_env(cfg, args.envs, seed=args.seed, precision="fp32", auto_reset=True)
    size = max(args.buffer, env.n_envs * max(args.collect_steps, 1))
    if args.prioritized:
        p = _priority_args(args)
        mem = S.PrioritizedReplayBuffer(size, (11,), 1, precision="fp32", device=local_rank, seed=args.seed + rank,
                                        as_torch=True, alpha=p["priority_alpha"], eps=p["priority_eps"])
    else:
        mem = S.ReplayBuffer(size, (11,), 1, precision="fp32", device=local_rank, seed=args.seed + rank, as_torch=True)
    agent = S.ContinuousAgent(cfg, exp.experiment_dir if exp else None, env.observation_space.shape, env,
                              device=local_rank, seed=args.seed + rank,
                              use_cuda_graph=not args.no_graph, memory=mem, policy_precision=args.policy_precision,
                              learner_precision=args.learner_precision, data_parallel=args.data_parallel or None,
                              **_algorithm_args(args), **(_priority_args(args) if args.prioritized else {}))
    act = agent.choose_action if args.no_graph else agent.choose_action_graphed
    obs = env.reset()
    rec = None
    if args.record_envs and exp:   # main.py:79: a recorder row every step; the ring holds a log interval (+ the first row)
        k = min(args.record_envs, env.n_envs)
        rec = S.DeviceRecorder(env, range(env.env_id_offset, env.env_id_offset + k), exp.experiment_dir,
                               capacity=max(1024, args.log_every + 1))
        rec.start()
    pipe = S.OverlappedActorLearner(agent, env, done_flag_mode=1, recorder=rec) if args.overlap else None
    losses = None
    rows, best, prev = [], float("-inf"), {"episodes": 0.0, "return_sum": 0.0}
    import random as _random
    pbt_prev, pbt_log, pbt_rng = {"episodes": 0.0, "return_sum": 0.0}, [], _random.Random(1000 + args.seed + rank)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(1, args.warmup_iters + args.iters + 1):
        if it == args.warmup_iters + 1:
            if pipe:
                pipe.finish()
            t0.record()
        if pipe:
            losses = pipe.step()
        elif args.collect_steps:
            agent.collect(env, args.collect_steps, done_flag_mode=1)   # T x (act, env.step, remember), one kernel
            for _ in range(args.updates_per_iter):
                out = agent.learn()
                losses = out if out is not None else losses
        else:
            actions = act(obs).squeeze(-1)
            agent.step_and_remember(env, actions, done_flag_mode=1)   # env.step + agent.remember, one kernel
            if rec:
                rec.capture(actions)
            for _ in range(args.updates_per_iter):
                out = agent.learn()
                losses = out if out is not None else losses
        if args.pbt_every and world > 1 and it % args.pbt_every == 0:
            if pipe:
                pipe.sync()
            c = env.counters()
            n = c["episodes"] - pbt_prev["episodes"]
            score = (c["return_sum"] - pbt_prev["return_sum"]) / n if n else float("nan")
            pbt_prev = c
            hp, info = S.population.exploit_explore(agent.training_tensors(), agent.hyperparameters(), score, pbt_rng)
            if info["adopted_from"] is not None:
                agent.set_hyperparameters(**hp)
                agent._weights_changed()
            pbt_log.append({"iter": it, "score": score, "adopted_from": info["adopted_from"], "hp": hp,
                            "ranking": info["ranking"]})
        if pipe and args.log_every and it % args.log_every == 0:
            pipe.sync()   # counters, losses and checkpoints below run on the default stream: order it after the pipeline
        if rec and args.log_every and it % args.log_every == 0:
            rec.flush()
        if args.data_parallel and args.experiments_root and args.log_every and it % args.log_every == 0:
            c = S.all_reduce_counters(env.counters_tensor())   # collective: the one agent's episodes on every rank
        if exp and args.log_every and it % args.log_every == 0:
            # one console.csv row per logging interval: the mean return of the episodes that ended in it
            if not args.data_parallel:
                c = env.counters()
            n = c["episodes"] - prev["episodes"]
            score = (c["return_sum"] - prev["return_sum"]) / n if n else float("nan")
            prev = c
            if n and score > best:
                best = score
                agent.save_models()          # main.py:104-106 keeps the checkpoints of improving episodes
            kind = max(S.TERM_NAMES[1:], key=lambda k: c[k])
            avg = c["return_sum"] / c["episodes"] if c["episodes"] else float("nan")
            rows.append([(rank, it), f"{kind}-{int(c[kind])}", score, best, avg, "", ""])
        if rank == 0 and args.log_every and it % args.log_every == 0:
            c = env.counters()
            lv = [float(x) for x in losses] if losses is not None else [float("nan")] * 3
            print(f"iter {it:6d}  episodes {c['episodes']:.0f}  goals {c['reached_goal']:.0f}  "
                  f"losses {_loss_label(args)} {lv[0]:.3g} {lv[1]:.3g} {lv[2]:.3g}", flush=True)
    if pipe:
        pipe.finish()
    t1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
    if world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    stats = S.all_reduce_counters(env.counters_tensor())
    if args.record_envs:
        recorded = torch.zeros(2, dtype=torch.float64, device="cuda")
        if rec:
            rec.close()
            recorded += torch.tensor([len(rec.ids), rec.episodes_finished], dtype=torch.float64, device="cuda")
        if world > 1:
            torch.distributed.all_reduce(recorded)
    sec = float(ms.item()) * 1e-3
    steps_per_iter = max(args.collect_steps, 1)
    summary = {"example": "train_sac", "overrides": overrides, "n_gpus": world, "envs_total": args.envs, "iters": args.iters,
               "updates_per_iter": args.updates_per_iter, "cuda_graph": not args.no_graph, "overlap": bool(args.overlap),
               "policy_precision": args.policy_precision, "learner_precision": args.learner_precision,
               "collect_steps": args.collect_steps,
               "env_steps_per_s": args.iters * steps_per_iter * args.envs / sec,
               "updates_per_s_per_replica": args.iters * args.updates_per_iter / sec,
               "ms_per_iter": 1e3 * sec / args.iters, "episodes": stats["episodes"],
               "mean_return": stats["return_mean"], "reached_goal": stats["reached_goal"],
               "losses_v_pi_q": [float(x) for x in losses] if losses is not None else None}
    if args.data_parallel:
        summary["data_parallel"], summary["effective_batch"] = True, world * agent.batch_size
    if args.algorithm == "sac2":
        summary["algorithm"], summary["temperature"] = "sac2", float(agent.temperature())
    if args.prioritized:
        summary["prioritized"] = True
        summary.update(_priority_args(args))
    if args.record_envs:   # over all ranks: envs recorded, and their episodes that ended (one info.csv row each)
        summary["recorded_envs"], summary["recorded_episodes"] = int(recorded[0]), int(recorded[1])
    if args.pbt_every:
        summary["pbt_rounds"] = len(pbt_log)
        summary["pbt_adoptions_rank0"] = [e for e in pbt_log if e["adopted_from"] is not None]
        summary["hyperparameters_rank0"] = agent.hyperparameters()
    if exp:
        c = stats if args.data_parallel else env.counters()
        exp.write_console(rows)
        exp.append_overview(best)
        exp.write_terminations(S.info_from_counters(c, max(S.TERM_NAMES[1:], key=lambda k: c[k])))
        summary["experiment_dir"], summary["best_interval_return"] = exp.experiment_dir, best
        if args.tune:
            summary["hpset"] = exp.tuner.hpset
        if world > 1 and not args.data_parallel:   # the population's best member, like reading overview.csv after a `-p` run
            scores = [None] * world
            torch.distributed.all_gather_object(scores, (best, rank, exp.experiment_name))
            summary["population_best"] = max(scores)
    if rank == 0:
        print(json.dumps(summary), flush=True)
    env.close(); mem.close()
    if world > 1 or args.data_parallel:
        torch.distributed.destroy_process_group()
    return summary


def _algorithm_args(args):
    """ContinuousAgent / AgentPopulation keyword arguments of --algorithm and the sac2 temperature flags."""
    if args.algorithm != "sac2":
        return {}
    return {"algorithm": "sac2", "target_entropy": args.target_entropy, "temperature_lr": args.temperature_lr,
            "init_temperature": 1.0 if args.init_temperature is None else args.init_temperature}


def _priority_args(args):
    """ContinuousAgent keyword arguments of --prioritized and the priority flags, their defaults filled in."""
    d = {"priority_alpha": 0.6, "priority_beta": 0.4, "priority_beta_updates": 0, "priority_eps": 1e-6}
    for k in d:
        if getattr(args, k) is not None:
            d[k] = type(d[k])(getattr(args, k))
    return {"prioritized": True, **d}


def _loss_label(args):
    return "t/pi/q" if args.algorithm == "sac2" else "v/pi/q"


def _overrides(args):
    out = {}
    for item in args.set:
        k, v = item.split("=", 1)
        out[k] = float(v) if any(ch in v for ch in ".e") else int(v)
    return out


def train_population(args, rank, local_rank, world, group=None):
    """--population P: P members per process (AgentPopulation), each trained as a replica would be.  With a process
    group (--data-parallel) every member is one agent trained by all ranks of `group` (rank and world are then this
    process's rank in it and its size): the ranks tune and rank the members alike, and rank 0 writes the experiments."""
    import random
    dp = group is not None
    torch.manual_seed(args.seed + rank)   # the Gaussian draws of the updates; each member's weights use seed + g
    P, overrides = args.population, _overrides(args)
    cfg = S.load_config(base_settings__experiment=args.experiment, **overrides)
    n_local = args.envs // world if dp else S.shard_range(args.envs, rank, world)[1]
    configs, exps = [cfg] * P, [None] * P
    if args.experiments_root:
        for m in range(P):
            g = rank * P + m
            if dp and rank > 0:   # rank 0's draw for member m, without writing its directory
                if args.tune:
                    configs[m] = S.AttrDict(S.HPTuner(rng=random.Random(args.seed + m)).tuned(cfg))
                continue
            exps[m] = S.Experiment(experiment_name=f"experiment_m{m}" if dp else f"experiment_r{rank}_m{m}",
                                   subdir=f"setting_{args.experiment}", root=args.experiments_root,
                                   rng=random.Random(args.seed + g))
            tuned = exps[m].save_configs(cfg)
            if args.tune:
                configs[m] = tuned
    pop = S.AgentPopulation(cfg, P, n_local, seed=args.seed, rank=rank, device=local_rank, configs=configs,
                            experiment_dirs=[e.experiment_dir if e else None for e in exps],
                            buffer_size=max(args.buffer, n_local * args.collect_steps),
                            data_parallel=group if dp else None, **_algorithm_args(args))
    pop.reset()
    losses = None
    rows, best = [[] for _ in range(P)], [float("-inf")] * P
    prev = [{"episodes": 0.0, "return_sum": 0.0} for _ in range(P)]
    pbt_prev = [{"episodes": 0.0, "return_sum": 0.0} for _ in range(P)]
    # data-parallel: one rng for every rank, so that all ranks make the same population rounds
    pbt_log, pbt_rng = [], random.Random(1000 + args.seed + (0 if dp else rank))

    def interval_score(c, p):
        n = c["episodes"] - p["episodes"]
        return (c["return_sum"] - p["return_sum"]) / n if n else float("nan")

    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(1, args.warmup_iters + args.iters + 1):
        if it == args.warmup_iters + 1:
            t0.record()
        pop.collect(args.collect_steps)
        for _ in range(args.updates_per_iter):
            out = pop.learn()
            losses = out if out is not None else losses
        if args.pbt_every and it % args.pbt_every == 0:
            counters = pop.counters()   # data-parallel: summed over the ranks
            scores = [interval_score(c, p) for c, p in zip(counters, pbt_prev)]
            pbt_prev = counters
            info = pop.exploit_explore(scores, pbt_rng)
            pbt_log.append({"iter": it, "scores": info["scores"], "ranking": info["ranking"],
                            "adopted": {m: {"from": info["best"], "hp": hp} for m, hp in info["adopted"].items()}})
        if args.log_every and it % args.log_every == 0:
            counters = pop.counters() if dp or args.experiments_root or rank == 0 else None
            for m, (a, exp) in enumerate(zip(pop.members, exps)):
                if exp is None:
                    continue
                c = counters[m]
                score = interval_score(c, prev[m])
                n = c["episodes"] - prev[m]["episodes"]
                prev[m] = c
                if n and score > best[m]:
                    best[m] = score
                    a.save_models()
                kind = max(S.TERM_NAMES[1:], key=lambda k: c[k])
                avg = c["return_sum"] / c["episodes"] if c["episodes"] else float("nan")
                rows[m].append([(rank, it), f"{kind}-{int(c[kind])}", score, best[m], avg, "", ""])
            if rank == 0:
                c = counters
                lv = [float(x) for x in losses[0]] if losses is not None else [float("nan")] * 3
                print(f"iter {it:6d}  episodes {sum(x['episodes'] for x in c):.0f}  goals "
                      f"{sum(x['reached_goal'] for x in c):.0f}  member 0 losses {_loss_label(args)} {lv[0]:.3g} "
                      f"{lv[1]:.3g} {lv[2]:.3g}", flush=True)
    t1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
    if world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX, group=group)
    total = torch.stack([env.counters_tensor() for env in pop.envs]).sum(0)
    stats = S.all_reduce_counters(total, group=group)
    final = pop.counters()   # data-parallel: summed over the ranks
    sec = float(ms.item()) * 1e-3
    members_total = P if dp else P * world
    summary = {"example": "train_sac", "overrides": overrides, "n_gpus": world, "envs_total": args.envs,
               "iters": args.iters, "updates_per_iter": args.updates_per_iter, "cuda_graph": not args.no_graph,
               "overlap": False, "policy_precision": args.policy_precision,
               "learner_precision": args.learner_precision, "collect_steps": args.collect_steps,
               "members": members_total, "members_per_gpu": P, "envs_per_member": n_local,
               "env_steps_per_s": args.iters * args.collect_steps * n_local * P * world / sec,
               "updates_per_s_per_replica": args.iters * args.updates_per_iter / sec,
               "updates_per_s_aggregate": args.iters * args.updates_per_iter * members_total / sec,
               "ms_per_iter": 1e3 * sec / args.iters, "episodes": stats["episodes"],
               "mean_return": stats["return_mean"], "reached_goal": stats["reached_goal"],
               "losses_v_pi_q": [[float(x) for x in l] for l in losses] if losses is not None else None}
    summary["env_steps_per_s_aggregate"] = summary["env_steps_per_s"]
    if dp:
        summary["data_parallel"], summary["effective_batch"] = True, world * pop.batch_size
    if args.algorithm == "sac2":
        summary["algorithm"], summary["temperature"] = "sac2", [float(a.temperature()) for a in pop.members]
    if args.pbt_every:
        summary["pbt_rounds"] = len(pbt_log)
        summary["pbt_adoptions"] = [e for e in pbt_log if e["adopted"]]
        summary["hyperparameters"] = [a.hyperparameters() for a in pop.members]
    if args.experiments_root and exps[0] is not None:
        for m, (a, exp) in enumerate(zip(pop.members, exps)):
            c = final[m]
            exp.write_console(rows[m])
            exp.append_overview(best[m])
            exp.write_terminations(S.info_from_counters(c, max(S.TERM_NAMES[1:], key=lambda k: c[k])))
        summary["experiment_dirs"] = [e.experiment_dir for e in exps]
        summary["best_interval_return"] = best
        if args.tune:
            summary["hpsets"] = [e.tuner.hpset for e in exps]
        mine = max((b, rank, e.experiment_name) for b, e in zip(best, exps))
        if world > 1 and not dp:
            scores = [None] * world
            torch.distributed.all_gather_object(scores, mine)
            mine = max(scores)
        summary["population_best"] = mine
    if rank == 0:
        print(json.dumps(summary), flush=True)
    pop.close()
    return summary


if __name__ == "__main__":
    main()
