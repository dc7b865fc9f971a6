#!/usr/bin/env python
"""Evaluation roll-outs on one GPU: the fused policy + env kernel (TensorCorePolicy.rollout, csrc/rollout.cu) against
the per-step loop it replaces (TensorCorePolicy.act, then BatchedBoatEnv.step without auto-reset), eager and replayed
from a CUDA graph of one step.

    python profiles/rollout_eval.py --out rollout_eval.json

Experiment 6, fp32, at 8192, 65,536 and 1,048,576 envs, two workloads:
  (a) the zero-mean-head actor, deterministic: every env runs straight to the goal (about 4960 steps);
  (b) a randomly initialised actor, stochastic, max_steps 1000 (episodes end at different steps).
The fused rollout is timed whole (CUDA events around the launch, after a reset).  The per-step loop runs every env
on every step until the last env's episode ends, so it is timed over that many steps -- in (a) over its first 500
steps, since every step does the same work, and scaled to the full length.  ms_per_step = time / steps of the
longest episode (all N envs per step); env_steps_per_s counts the steps envs actually take before their episode
ends (the sum of steps_out), for both paths.  Variants alternate over the repetitions and the median is kept.
With --pair-library, the fused kernel's grid (one 128-env tile per CTA while tiles < SMs) is timed against two tiles
per CTA at 8192 and 65,536 envs, each build in fresh processes, alternating.  The
share of the piece-change setup is not separable: it runs inside the env step of the fused kernel.  The card's name
and power limit are read in the same run.  One JSON document, printed and written to --out.
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
    if kind == "zero_mean":
        with torch.no_grad():
            net.mean.weight.zero_()
            net.mean.bias.zero_()
    return net


def workload(n, kind, deterministic, max_steps, loop_steps, reps, fused_only=False):
    cfg = S.load_config(base_settings__experiment=6)
    env = S.BatchedBoatEnv(cfg, n, seed=0, precision="fp32", device=0, auto_reset=False)
    pol = TensorCorePolicy(actor(kind), seed=3)
    eps = torch.zeros((n, 1), dtype=torch.float32, device=env.device) if deterministic else None

    def fused():
        env.reset()
        out = {}
        out["ms"] = timed(lambda: out.setdefault("r", pol.rollout(env, max_steps, deterministic)))
        return out

    first = fused()   # warm-up; also tells how long the longest episode is
    steps = first["r"][1]
    longest, env_steps = int(steps.max()), int(steps.sum())
    n_loop = min(loop_steps or longest, longest)
    if fused_only:
        ms = [fused()["ms"] for _ in range(reps)]
        env.close()
        return {"envs": n, "actor": kind, "longest_episode": longest, "fused_ms": statistics.median(ms), "samples_ms": ms}

    def step_once():
        a = pol.act(env.obs, eps=eps)
        env.step(a.reshape(-1))

    def eager():
        env.reset()
        return timed(lambda: [step_once() for _ in range(n_loop)])

    env.reset()
    step_once()   # warm-up of both kernels before the capture
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step_once()
        with torch.cuda.graph(g, stream=s):
            step_once()
    torch.cuda.current_stream().wait_stream(s)

    def graphed():
        env.reset()
        return timed(lambda: [g.replay() for _ in range(n_loop)])

    eager()
    graphed()
    res = {"fused": [], "eager_loop": [], "graph_loop": []}
    for _ in range(reps):
        res["fused"].append(fused()["ms"])
        res["eager_loop"].append(eager() * longest / n_loop)
        res["graph_loop"].append(graphed() * longest / n_loop)
    out = {"envs": n, "actor": kind, "deterministic": deterministic, "max_steps": max_steps,
           "longest_episode": longest, "env_steps": env_steps, "loop_steps_timed": n_loop,
           "terminations": {S.TERM_NAMES[k]: int((first["r"][2] == k).sum()) for k in range(1, 6)}}
    for k, v in res.items():
        ms = statistics.median(v)
        out[k] = {"ms": ms, "ms_per_step": ms / longest, "env_steps_per_s": env_steps / (ms * 1e-3), "samples_ms": v}
    out["speedup_vs_graph_loop"] = out["graph_loop"]["ms"] / out["fused"]["ms"]
    out["speedup_vs_eager_loop"] = out["eager_loop"]["ms"] / out["fused"]["ms"]
    env.close()
    del g
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="8192,65536,1048576")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pair-library", default=None,
                    help="a libboatenv build with -DBOAT_ROLLOUT_PAIR_TILES (python -m sac_agent_b200._build --variant "
                         "pair -DBOAT_ROLLOUT_PAIR_TILES): the fused kernel's grid choice is timed against it")
    ap.add_argument("--fused-only", action="store_true", help="(internal) time the fused kernel only, print one JSON line")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "rollout_eval needs a GPU"
    torch.cuda.set_device(0)
    if args.fused_only:
        rows = [workload(int(x), k, d, m, 0, args.reps, fused_only=True) for x in args.sizes.split(",")
                for k, d, m in (("zero_mean", True, 6000), ("random_init", False, 1000))]
        print(json.dumps({"library": S.library_path(), "rows": rows}))
        return
    doc = {"card": card(), "experiment": 6, "precision": "fp32", "workloads": []}
    for n in [int(x) for x in args.sizes.split(",")]:
        doc["workloads"].append(workload(n, "zero_mean", True, 6000, 500, args.reps))
        doc["workloads"].append(workload(n, "random_init", False, 1000, 0, args.reps))
        w = doc["workloads"][-2:]
        print(json.dumps({"envs": n, "a_speedup_vs_graph": w[0]["speedup_vs_graph_loop"],
                          "b_speedup_vs_graph": w[1]["speedup_vs_graph_loop"]}), flush=True)
    if args.pair_library:
        # the grid choice below 2 x SMs tiles: one tile per CTA (this build) against two per CTA, in fresh processes,
        # alternating
        runs = {"one_tile_per_cta": [], "two_tiles_per_cta": []}
        for _ in range(2):
            for name, lib in (("one_tile_per_cta", None), ("two_tiles_per_cta", args.pair_library)):
                env = dict(os.environ)
                env.pop("BOATENV_LIBRARY", None)
                if lib:
                    env["BOATENV_LIBRARY"] = os.path.abspath(lib)
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--fused-only", "--sizes", "8192,65536",
                                      "--reps", "3"], env=env, capture_output=True, text=True, check=True).stdout
                runs[name].append(json.loads(out.strip().splitlines()[-1]))
        doc["grid_choice"] = runs
        for name, rr in runs.items():
            print(name, [[round(r["fused_ms"], 3) for r in run["rows"]] for run in rr], flush=True)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
