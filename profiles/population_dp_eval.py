#!/usr/bin/env python
"""Data-parallel population updates against the fused ones, on one GPU over a one-rank NCCL group.  Per round of P
members at B = 1024:
  (a) AgentPopulation.learn(): boatreplay_sample_members + one normal_ + boatagent_sac_update_members (two launches);
  (b) AgentPopulation(data_parallel=group).learn(): the same gather and draw, boatagent_sac_gradients_members (two
      launches), one all-reduce of the [P, n_params + 3] gradient buffer, boatagent_adam_polyak_members (one launch);
  (c) P data-parallel ContinuousAgents, learn() one after another on one stream (per member: gather, draw,
      boatagent_sac_gradients, all-reduce, boatagent_adam_polyak_step).
P in {1, 2, 4, 8, 16}, CUDA events over 50 rounds, median of 7 repetitions alternating the arms.  Before timing,
(a) and (b) are built from the same seeds and compared bit for bit over three rounds with the same Gaussian draws.
World sizes 2, 4 and 8 need that many GPUs and are recorded as not measured otherwise.

    python profiles/population_dp_eval.py [--out profiles/population_dp_eval.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sac_agent_b200 as S  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def timed(fn, rounds):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / rounds


def state(pop):
    out = []
    for a in pop.members:
        o = a.learner.optimizer
        out += [p.data for net in a.learner.networks() for p in net.parameters()] + [p.grad for p in o.params]
        out += o.state_tensors() + [a._loss_buf]
    return out


def identical(fused, split, rounds=3):
    """Three rounds of both populations on the same rings and the same Gaussian draws, compared bit for bit."""
    for _ in range(rounds):
        rng = torch.cuda.get_rng_state()
        fused.learn()
        torch.cuda.set_rng_state(rng)
        split.learn()
    torch.cuda.synchronize()
    return all(torch.equal(x, y) for x, y in zip(state(fused), state(split)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "population_dp_eval.json"))
    ap.add_argument("--sizes", default="1,2,4,8,16")
    ap.add_argument("--rounds", type=int, default=50)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1, device_id=torch.device("cuda", 0))
    group = dist.group.WORLD
    n_gpus = torch.cuda.device_count()
    res = {"gpu": card(), "batch": 1024, "world": 1, "backend": "nccl", "rounds": args.rounds, "reps": args.reps,
           "learn": [], "world_2_4_8": f"not measured ({n_gpus} GPU visible)"}
    cfg = S.load_config(base_settings__experiment=5)
    for P in [int(x) for x in args.sizes.split(",")]:
        fused = S.AgentPopulation(cfg, P, 1024, seed=0, buffer_size=65536)
        split = S.AgentPopulation(cfg, P, 1024, seed=0, buffer_size=65536, data_parallel=group)
        for pop in (fused, split):
            pop.reset()
            pop.collect(2)   # 2048 rows per ring: more than a batch
        same = identical(fused, split)
        agents, envs = [], []
        for m in range(P):
            env = S.BatchedBoatEnv(cfg, 1024, seed=0, precision="fp32", device=0, env_id_offset=m * 1024)
            mem = S.ReplayBuffer(65536, (11,), 1, precision="fp32", device=0, seed=m, as_torch=True)
            torch.manual_seed(m)
            a = S.ContinuousAgent(cfg, None, env.observation_space.shape, env, device=0, seed=m, memory=mem,
                                  policy_precision="tcgen05", learner_precision="tcgen05", data_parallel=group)
            env.reset()
            a.collect(env, 2)
            agents.append(a)
            envs.append(env)

        def arm_c():
            for a in agents:
                a.learn()

        arms = {"a_fused_population": fused.learn, "b_data_parallel_population": split.learn,
                "c_data_parallel_agents_one_stream": arm_c}
        for fn in arms.values():   # warm-up
            timed(fn, 5)
        ms = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, fn in arms.items():
                ms[k].append(timed(fn, args.rounds))
        row = {"members": P, **{k + "_ms": statistics.median(v) for k, v in ms.items()},
               "spread": {k: [min(v), max(v)] for k, v in ms.items()}, "a_b_bit_identical": same}
        row["b_over_a"] = row["b_data_parallel_population_ms"] / row["a_fused_population_ms"]
        row["b_aggregate_updates_per_s"] = 1e3 * P / row["b_data_parallel_population_ms"]
        row["c_aggregate_updates_per_s"] = 1e3 * P / row["c_data_parallel_agents_one_stream_ms"]
        row["b_over_c_updates_per_s"] = row["b_aggregate_updates_per_s"] / row["c_aggregate_updates_per_s"]
        res["learn"].append(row)
        print(json.dumps(row), flush=True)
        for pop in (fused, split):
            pop.close()
        for a, env in zip(agents, envs):
            env.close()
            a.memory.close()
        del fused, split, agents, envs
        torch.cuda.empty_cache()
    dist.destroy_process_group()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "wrote": args.out}))


if __name__ == "__main__":
    main()
