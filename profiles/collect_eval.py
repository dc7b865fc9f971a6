#!/usr/bin/env python
"""Experience collection on one GPU: the fused act + step + remember kernel (TensorCorePolicy.collect, csrc/rollout.cu)
against the loop examples/train_sac.py runs without --collect-steps (TensorCorePolicy.act, then ReplayBuffer.step_store
on the auto-resetting env: two launches per step, eager).

    python profiles/collect_eval.py --out collect_eval.json

Experiment 6, fp32, a 2^24-slot ring (16.7 M rows, 1.6 GB), two actors:
  random_init  a seeded default init: an episode ends about every 140 steps, so envs reset inside the kernel often;
  low_noise    mean head zero, log_std -5: long episodes, almost no resets.
Sizes: 8192 and 65,536 envs with T = 256 steps per call, 1,048,576 envs with T = 16.  Both paths start from the same
fresh envs and rings; their first call is compared bit for bit (ring rows, observations, rewards, termination codes,
env state) and the timed calls follow, alternating between the two paths; medians are reported.  ms_per_step is the
time of a call over T (every env steps every step).

--driver also times examples/train_sac.py at 8192 envs: --collect-steps 8 --updates-per-iter 8 against the per-step
loop with one update per step (the same update-to-data ratio, tcgen05 acting in both), as ms per env step.
The card's name and power limit are read in the same run.  One JSON document, printed and written to --out.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200.networks import ActorNetwork, TensorCorePolicy  # noqa: E402

RING = 1 << 24
COUNTER_BYTES = 32 * 32 * 8


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:  # reported, not guessed
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def actor(kind):
    torch.manual_seed(1)
    net = ActorNetwork(None, (11,), max_action=[1.0]).cuda()
    if kind == "low_noise":
        with torch.no_grad():
            net.mean.weight.zero_()
            net.mean.bias.zero_()
            net.std.bias.fill_(-20.0)
    return net


def same(x, y):
    if x.dtype == torch.float32:
        x, y = x.contiguous().view(torch.int32), y.contiguous().view(torch.int32)
    return bool(torch.equal(x, y))


def rows(mem, first, count):
    idx = (torch.arange(count, dtype=torch.int64, device=mem.device) + first) % mem.mem_size
    return mem.gather(idx, as_torch=True)


def workload(n, T, kind, reps):
    cfg = S.load_config(base_settings__experiment=6)
    net = actor(kind)
    paths = {}
    for name in ("fused", "loop"):
        env = S.BatchedBoatEnv(cfg, n, seed=0, precision="fp32", device=0, auto_reset=True)
        env.reset()
        mem = S.ReplayBuffer(RING, (11,), 1, precision="fp32", device=0, as_torch=True)
        paths[name] = (env, mem, TensorCorePolicy(net, seed=3))

    def fused():
        env, mem, pol = paths["fused"]
        pol.collect(env, mem, T)

    def loop():
        env, mem, pol = paths["loop"]
        for _ in range(T):
            a = pol.act(env.obs)
            mem.step_store(env, a.reshape(-1))

    # first call of each path: warm-up and the output comparison
    fused()
    loop()
    torch.cuda.synchronize()
    (ef, mf, _), (ee, me, _) = paths["fused"], paths["loop"]
    rf, re_ = rows(mf, 0, T * n), rows(me, 0, T * n)
    check = {"ring": all(same(x, y) for x, y in zip(rf, re_)),
             "obs_reward_term": same(ef.obs, ee.obs) and same(ef.reward, ee.reward) and same(ef.term, ee.term),
             "env_state": same(ef.state_dict()["blob"][:-COUNTER_BYTES], ee.state_dict()["blob"][:-COUNTER_BYTES])}
    del rf, re_
    episodes = ef.counters()["episodes"]
    res = {"fused": [], "loop": []}
    for _ in range(reps):
        res["fused"].append(timed(fused))
        res["loop"].append(timed(loop))
    out = {"envs": n, "steps_per_call": T, "actor": kind, "bit_identical": check,
           "episodes_ended_in_first_call": episodes, "resets_per_env_step": episodes / (n * T)}
    for k, v in res.items():
        ms = statistics.median(v)
        out[k] = {"ms": ms, "ms_per_step": ms / T, "env_steps_per_s": n * T / (ms * 1e-3), "samples_ms": v}
    out["speedup"] = out["loop"]["ms"] / out["fused"]["ms"]
    for env, mem, _ in paths.values():
        env.close()
        mem.close()
    return out


def driver(reps):
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import train_sac
    common = ["--envs", "8192", "--experiment", "6", "--policy-precision", "tcgen05", "--log-every", "0"]
    runs = {"per_step": [], "collect8": []}
    for _ in range(reps):
        s = train_sac.main(common + ["--iters", "400", "--warmup-iters", "40", "--updates-per-iter", "1"])
        runs["per_step"].append(s["ms_per_iter"])
        s = train_sac.main(common + ["--iters", "50", "--warmup-iters", "5", "--collect-steps", "8",
                                     "--updates-per-iter", "8"])
        runs["collect8"].append(s["ms_per_iter"] / 8)
    out = {"envs": 8192, "experiment": 6, "per_step": {"ms_per_env_step": statistics.median(runs["per_step"]),
                                                       "samples": runs["per_step"]},
           "collect8": {"ms_per_env_step": statistics.median(runs["collect8"]), "samples": runs["collect8"]}}
    out["speedup"] = out["per_step"]["ms_per_env_step"] / out["collect8"]["ms_per_env_step"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="8192:256,65536:256,1048576:16", help="envs:steps per call, comma separated")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--driver", action="store_true", help="also time examples/train_sac.py (see the module doc)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "collect_eval needs a GPU"
    torch.cuda.set_device(0)
    doc = {"card": card(), "experiment": 6, "precision": "fp32", "ring_slots": RING, "workloads": []}
    for item in args.sizes.split(","):
        n, T = (int(x) for x in item.split(":"))
        for kind in ("random_init", "low_noise"):
            w = workload(n, T, kind, args.reps)
            doc["workloads"].append(w)
            print(json.dumps({k: w[k] for k in ("envs", "actor", "bit_identical", "speedup")}), flush=True)
    if args.driver:
        doc["train_sac"] = driver(3)
        print(json.dumps(doc["train_sac"]), flush=True)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
