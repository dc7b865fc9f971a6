#!/usr/bin/env python
"""Population updates on one GPU: P members' update rounds as (a) P ContinuousAgent.learn() calls on one stream,
(b) the same calls on P streams, (c) one AgentPopulation.learn() (boatreplay_sample_members + one normal_ +
boatagent_sac_update_members).  B = 1024, P in {1, 2, 4, 8, 16}, CUDA events over 50 rounds, median of 7 alternating
repetitions.  At every size, (c)'s update is checked bit for bit against each member's own boatagent_sac_update on the
same batch and draws.  Then train_sac --population P at 8192 envs per member, collect 8 + 8 updates per iteration.

    python profiles/population_eval.py [--out profiles/population_eval.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
import sac_agent_b200 as S  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def state(a):
    o = a.learner.optimizer
    return ([p.data for net in a.learner.networks() for p in net.parameters()] + [p.grad for p in o.params]
            + o.state_tensors() + [a._loss_buf])


def identical(pop):
    """pop.learn() against each member's own boatagent_sac_update on the batch and draws it used."""
    before = [[t.clone() for t in state(a)] for a in pop.members]
    pop.learn()
    after = [[t.clone() for t in state(a)] for a in pop.members]
    for a, st in zip(pop.members, before):
        with torch.no_grad():
            torch._foreach_copy_(state(a), st)
        a._fused_update()
    torch.cuda.synchronize()
    return all(torch.equal(x, y) for a, ref in zip(pop.members, after) for x, y in zip(state(a), ref))


def timed(fn, rounds):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / rounds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "population_eval.json"))
    ap.add_argument("--sizes", default="1,2,4,8,16")
    ap.add_argument("--rounds", type=int, default=50)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--train-iters", type=int, default=30)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"gpu": card(), "batch": 1024, "rounds": args.rounds, "reps": args.reps, "learn": [], "train_sac": []}
    cfg = S.load_config(base_settings__experiment=5)
    for P in [int(x) for x in args.sizes.split(",")]:
        pop = S.AgentPopulation(cfg, P, 1024, seed=0, buffer_size=65536)
        pop.reset()
        pop.collect(2)   # 2048 rows per ring: more than a batch
        streams = [torch.cuda.Stream() for _ in range(P)]

        def arm_a():
            for a in pop.members:
                a.learn()

        def arm_b():
            cur = torch.cuda.current_stream()
            for a, s in zip(pop.members, streams):
                s.wait_stream(cur)
                with torch.cuda.stream(s):
                    a.learn()
            for s in streams:
                cur.wait_stream(s)

        arms = {"a_solo_one_stream": arm_a, "b_solo_p_streams": arm_b, "c_population": pop.learn}
        for fn in arms.values():   # warm-up
            timed(fn, 5)
        ms = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, fn in arms.items():
                ms[k].append(timed(fn, args.rounds))
        row = {"members": P, **{k + "_ms": statistics.median(v) for k, v in ms.items()},
               "spread": {k: [min(v), max(v)] for k, v in ms.items()}, "c_bit_identical_to_solo": identical(pop)}
        row["c_aggregate_updates_per_s"] = 1e3 * P / row["c_population_ms"]
        res["learn"].append(row)
        print(json.dumps(row), flush=True)
        pop.close()
        del pop
        torch.cuda.empty_cache()
    solo = res["learn"][0]["c_population_ms"]
    for row in res["learn"]:
        row["c_round_over_solo_update"] = row["c_population_ms"] / solo
    import train_sac
    for P in [int(x) for x in args.sizes.split(",")]:
        s = train_sac.main(["--envs", "8192", "--population", str(P), "--policy-precision", "tcgen05",
                            "--learner-precision", "tcgen05", "--collect-steps", "8", "--updates-per-iter", "8",
                            "--iters", str(args.train_iters), "--warmup-iters", "5", "--log-every", "0",
                            "--buffer", "262144"])
        row = {k: s[k] for k in ("members", "ms_per_iter", "env_steps_per_s_aggregate", "updates_per_s_aggregate")}
        res["train_sac"].append(row)
        print(json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    base = res["train_sac"][0]
    for row in res["train_sac"]:
        row["updates_per_s_vs_p1"] = row["updates_per_s_aggregate"] / base["updates_per_s_aggregate"]
        row["env_steps_per_s_vs_p1"] = row["env_steps_per_s_aggregate"] / base["env_steps_per_s_aggregate"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "wrote": args.out}))


if __name__ == "__main__":
    main()
