#!/usr/bin/env python
"""SAC-v2 (ContinuousAgent(algorithm="sac2")) against SAC-v1, per update, on one GPU.

    python profiles/sac2_eval.py --out sac2_eval.json

Per update, at B = 256, 1024 and 4096: four agents -- v1 fp32 graph, v1 fused tcgen05, v2 fp32 graph, v2 fused
tcgen05 -- each replaying its update on one fixed batch, timed with CUDA events over 50 updates, alternating between
the four arms for 7 rounds after warm-up; medians are reported.  Batch and weights are a few MB, so every arm runs from
L2.  Before the timing, one fused v2 update on that batch is checked against the bf16 emulation of tests/test_sac2.py
(its tolerance).  Then one v2 population round (FusedLearner over P members, three launches) at B = 1024 for
P = 1, 4, 8 and 16, timed the same way.  The card's name and power limit are read in the same run.  Targets: the fused
v2 update at B = 1024 no slower than the fused v1 update, and faster than the v2 fp32 graph.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import torch  # noqa: E402

import test_gpu_learner as T1  # noqa: E402
import test_sac2 as T2  # noqa: E402
from learner_eval import card, timed  # noqa: E402
from sac_agent_b200.continuous_agent import FusedLearner  # noqa: E402


def _load(agent, b):
    for dst, src in zip(agent._batch, (b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8))):
        dst.copy_(src.reshape(dst.shape))
    agent._eps.copy_(b["eps"])


def per_update(B, rounds=7, n=50):
    b = T2._batch(B, B, "cuda")
    agents = {"v1_fp32_graph": T1._agent(B, learner_precision="fp32", seed=B),
              "v1_fused": T1._agent(B, learner_precision="tcgen05", seed=B),
              "v2_fp32_graph": T2._agent(B, "fp32", seed=B),
              "v2_fused": T2._agent(B, "tcgen05", seed=B)}
    T2._away_from_init(agents["v2_fused"], B)
    worst = T2._check_update(agents["v2_fused"], b)   # asserts the test's tolerances
    for a in agents.values():
        _load(a, b)
        for _ in range(10):   # warm-up; the fp32 learners capture their graphs here
            a._run_update()
    torch.cuda.synchronize()
    times = {k: [] for k in agents}
    for _ in range(rounds):
        for k, a in agents.items():
            times[k].append(timed(a._run_update, n))
    for a in agents.values():
        a.memory.close()
    med = {k: statistics.median(t) for k, t in times.items()}
    return {"batch": B, "ms_per_update": med, "all_ms": times,
            "v2_fused_vs_emulation_worst_grad_err": max(worst.values()),
            "v2_fused_vs_emulation_worst_tensor": max(worst, key=worst.get)}


def population(P, B=1024, rounds=7, n=50):
    members = [T2._agent(B, "tcgen05", seed=100 + m) for m in range(P)]
    for m, a in enumerate(members):
        _load(a, T2._batch(B, 1000 * P + m, "cuda"))
    fl = FusedLearner(members)
    for _ in range(10):
        fl.update()
    torch.cuda.synchronize()
    t = [timed(fl.update, n) for _ in range(rounds)]
    for a in members:
        a.memory.close()
    return {"members": P, "batch": B, "ms_per_round": statistics.median(t), "all_ms": t,
            "ms_per_member_update": statistics.median(t) / P}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "sac2_eval needs the GPU"
    out = {"card": card(), "per_update": [per_update(B) for B in (256, 1024, 4096)],
           "population_v2": [population(P) for P in (1, 4, 8, 16)]}
    at1024 = next(r for r in out["per_update"] if r["batch"] == 1024)["ms_per_update"]
    out["targets"] = {
        "v2_fused_no_slower_than_v1_fused_at_1024": {"v2_fused_ms": at1024["v2_fused"], "v1_fused_ms": at1024["v1_fused"],
                                                     "met": at1024["v2_fused"] <= at1024["v1_fused"]},
        "v2_fused_faster_than_v2_fp32_graph_at_1024": {"v2_fused_ms": at1024["v2_fused"],
                                                       "v2_fp32_graph_ms": at1024["v2_fp32_graph"],
                                                       "met": at1024["v2_fused"] < at1024["v2_fp32_graph"]}}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
