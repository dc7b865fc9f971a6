#!/usr/bin/env python
"""What recording costs inside the fused collection kernel: TensorCorePolicy.collect with a DeviceRecorder
(boatagent_collect_record, csrc/rollout.cu) against plain collect, and against the per-step loop that was the only
way to record before (TensorCorePolicy.act, ReplayBuffer.step_store, DeviceRecorder.capture: three launches a step).

    python profiles/collect_record_eval.py --out collect_record_eval.json

Experiment 6, fp32, a 2^24-slot replay ring, the seeded random-init actor of collect_eval.py (an env resets about
every 72 env-steps).  Sizes: 8192 and 65,536 envs with T = 256 steps per call, 1,048,576 envs with T = 16.  Paths,
each on its own fresh env and ring:
  plain     collect(T)
  rec64     collect(T, recorder=...) recording M = 64 envs spread over the population
  rec1024   the same with M = 1024
  loop64    T rounds of act + step_store + capture() with M = 64
Recorder capacity is T and the pending rows are dropped unwritten between calls, so no timed call contains a flush:
the numbers are the GPU work.  The first call of each path is the warm-up and the output check: rec64's recorder
ring equals loop64's bit for bit (all ten columns), and rec64's replay ring, observations and env state equal
plain's.  Then `--reps` timed calls per path, alternating between the paths; medians of CUDA-event times.

--train also times a training loop at 8192 envs: agent.collect(env, 8) plus 8 learn() calls per iteration, with a
DeviceRecorder of 64 envs flushed (CSV files written) every 50 iterations, against the same loop without a recorder;
rec64_unwritten drops the rows every 50 iterations instead of writing them (the GPU and launch cost alone).
The card's name and power limit are read in the same run.  One JSON document, printed and written to --out.
"""
import argparse
import json
import os
import statistics
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sac_agent_b200 as S  # noqa: E402
from collect_eval import RING, COUNTER_BYTES, actor, card, rows, same, timed  # noqa: E402
from sac_agent_b200.networks import TensorCorePolicy  # noqa: E402

COLUMNS = ("s_x", "s_y", "v_x", "v_y", "s_r", "rudder_angle", "action", "reward", "term", "episode")


def drop_pending(rec):
    """Forgets the recorder's pending rows without writing them (the timed calls measure the GPU work only)."""
    rec._flushed = rec._rows
    del rec._stepped[:]


def workload(n, T, reps, tmp):
    cfg = S.load_config(base_settings__experiment=6)
    net = actor("random_init")
    rng = np.random.default_rng(n)
    ids = {64: [int(i) for i in rng.choice(n, 64, replace=False)],
           1024: [int(i) for i in rng.choice(n, 1024, replace=False)]}
    paths = {}
    for name, m in (("plain", 0), ("rec64", 64), ("rec1024", 1024), ("loop64", 64)):
        env = S.BatchedBoatEnv(cfg, n, seed=0, precision="fp32", device=0, auto_reset=True)
        env.reset()
        mem = S.ReplayBuffer(RING, (11,), 1, precision="fp32", device=0, as_torch=True)
        rec = S.DeviceRecorder(env, ids[m], os.path.join(tmp, f"{n}_{name}"), capacity=T) if m else None
        paths[name] = (env, mem, TensorCorePolicy(net, seed=3), rec)

    def run(name):
        env, mem, pol, rec = paths[name]
        if rec is not None:
            drop_pending(rec)
        if name == "loop64":
            for _ in range(T):
                a = pol.act(env.obs).reshape(-1)
                mem.step_store(env, a)
                rec.capture(a)
        else:
            pol.collect(env, mem, T, recorder=rec)

    for name in paths:   # first call of each path: warm-up and the output check
        run(name)
    torch.cuda.synchronize()
    (ep, mp, _, _), (er, mr, _, rr), (_, _, _, rl) = paths["plain"], paths["rec64"], paths["loop64"]
    check = {"recorder_ring_vs_loop64": all(same(rr._cols[k], rl._cols[k]) for k in COLUMNS),
             "replay_ring_vs_plain": all(same(x, y) for x, y in zip(rows(mr, 0, T * n), rows(mp, 0, T * n))),
             "obs_reward_term_vs_plain": same(er.obs, ep.obs) and same(er.reward, ep.reward) and same(er.term, ep.term),
             "env_state_vs_plain": same(er.state_dict()["blob"][:-COUNTER_BYTES],
                                        ep.state_dict()["blob"][:-COUNTER_BYTES])}
    recorded_ends = int(rr._cols["term"].ne(0).sum())
    res = {name: [] for name in paths}
    for _ in range(reps):
        for name in paths:
            res[name].append(timed(lambda: run(name)))
    out = {"envs": n, "steps_per_call": T, "bit_identical": check, "recorded_episode_ends_in_first_call": recorded_ends}
    for name, v in res.items():
        ms = statistics.median(v)
        out[name] = {"ms": ms, "ms_per_step": ms / T, "samples_ms": v}
    for name in ("rec64", "rec1024", "loop64"):
        out[name]["overhead_vs_plain_pct"] = 100.0 * (out[name]["ms"] / out["plain"]["ms"] - 1.0)
    out["loop64_over_rec64"] = out["loop64"]["ms"] / out["rec64"]["ms"]
    for env, mem, _, rec in paths.values():
        if rec is not None:
            drop_pending(rec)
            rec.close()
        env.close()
        mem.close()
    return out


def train_loop(reps, iters, tmp):
    from sac_agent_b200 import ContinuousAgent
    cfg = S.load_config(base_settings__experiment=6)
    n, T, updates, flush_every = 8192, 8, 8, 50
    runs = {}
    for name in ("plain", "rec64", "rec64_unwritten"):
        torch.manual_seed(5)
        env = S.BatchedBoatEnv(cfg, n, seed=1, precision="fp32", device=0, auto_reset=True)
        mem = S.ReplayBuffer(1 << 20, (11,), 1, precision="fp32", device=0, as_torch=True)
        agent = ContinuousAgent(cfg, None, (11,), env, device=0, seed=1, memory=mem, policy_precision="tcgen05")
        env.reset()
        rec = None
        if name != "plain":
            ids = [int(i) for i in np.random.default_rng(2).choice(n, 64, replace=False)]
            rec = S.DeviceRecorder(env, ids, os.path.join(tmp, "train_" + name), capacity=T * flush_every + 1)
            rec.start()
        runs[name] = (env, agent, rec)

    def run(name):
        env, agent, rec = runs[name]
        for it in range(iters):
            agent.collect(env, T, recorder=rec)
            for _ in range(updates):
                agent.learn()
            if rec is not None and (it + 1) % flush_every == 0:
                rec.flush() if name == "rec64" else drop_pending(rec)

    for name in runs:
        run(name)   # warm-up: graphs, fill the ring past the batch size
    res = {name: [] for name in runs}
    for _ in range(reps):
        for name in runs:
            res[name].append(timed(lambda: run(name)) / (iters * T))
    out = {"envs": n, "collect_steps": T, "updates_per_iter": updates, "iters_per_sample": iters,
           "recorded_envs": 64, "flush_every_iters": flush_every}
    for name, v in res.items():
        out[name] = {"ms_per_env_step": statistics.median(v), "samples": v}
    for name in ("rec64", "rec64_unwritten"):
        out[name]["overhead_vs_plain_pct"] = 100.0 * (out[name]["ms_per_env_step"] / out["plain"]["ms_per_env_step"] - 1)
    out["recorded_episodes"] = runs["rec64"][2].episodes_finished
    for env, _, rec in runs.values():
        if rec is not None:
            rec.close()
        env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="8192:256,65536:256,1048576:16", help="envs:steps per call, comma separated")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--train", action="store_true", help="also time the training loop (see the module doc)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "collect_record_eval needs a GPU"
    torch.cuda.set_device(0)
    doc = {"card": card(), "experiment": 6, "precision": "fp32", "ring_slots": RING, "actor": "random_init",
           "target": "rec64 at most +2 % over plain collect", "workloads": []}
    with tempfile.TemporaryDirectory() as tmp:
        for item in args.sizes.split(","):
            n, T = (int(x) for x in item.split(":"))
            w = workload(n, T, args.reps, tmp)
            doc["workloads"].append(w)
            print(json.dumps({k: w[k] for k in ("envs", "bit_identical")} |
                             {p: round(w[p]["overhead_vs_plain_pct"], 2) for p in ("rec64", "rec1024", "loop64")}),
                  flush=True)
        doc["target_met"] = all(w["rec64"]["overhead_vs_plain_pct"] <= 2.0 for w in doc["workloads"])
        if args.train:
            doc["train_loop"] = train_loop(5, 100, tmp)
            print(json.dumps(doc["train_loop"]), flush=True)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
