#!/usr/bin/env python
"""Prioritized experience replay (PrioritizedReplayBuffer, ContinuousAgent(prioritized=True)) against uniform replay,
on one GPU.

    python profiles/per_eval.py --out per_eval.json

1. sample + gather: PrioritizedReplayBuffer.sample_buffer (stratified draw, weights, boatreplay_gather) against
   ReplayBuffer.sample_buffer (boatreplay_sample) into a static batch, at B = 1024 and 4096, on full rings of 2^20 and
   2^25 slots (the 2^25 ring and its 128 MB of leaves are larger than the 126 MB L2).
2. update_priorities at B = 1024 and 4096, and fill_new of the 8192 x 8 rows one collect stores.
3. one learn() (the draw, the update and, prioritized, the priority update) against a uniform learn(), for SAC-v1 and
   SAC-v2 with the fp32 graph and the fused tcgen05 learner, at B = 1024 on a full 2^25 ring.
4. the train_sac loop at 8192 envs, --collect-steps 8 --updates-per-iter 8, fused learner, with and without
   --prioritized (device-timed iterations per second from its summary).
Every arm is timed with CUDA events over many calls, alternating between arms for several rounds after warm-up;
medians are reported.  The card's name and power limit are read in the same run.
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, os.path.join(os.path.dirname(ROOT), "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(ROOT), "examples"))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import sac_agent_b200 as S  # noqa: E402
from boat_testlib import set_mem_cntr  # noqa: E402
from learner_eval import card, timed  # noqa: E402
from sac_agent_b200.continuous_agent import ContinuousAgent  # noqa: E402
from test_gpu_learner import _env_stub  # noqa: E402


def alternate(arms, rounds, n):
    for f in arms.values():
        for _ in range(5):
            f()
    torch.cuda.synchronize()
    t = {k: [] for k in arms}
    for _ in range(rounds):
        for k, f in arms.items():
            t[k].append(timed(f, n))
    return {k: statistics.median(v) for k, v in t.items()}, t


def rings(log2):
    n = 1 << log2
    uni = S.ReplayBuffer(n, (11,), 1, precision="fp32", device=0, seed=1, as_torch=True)
    per = S.PrioritizedReplayBuffer(n, (11,), 1, precision="fp32", device=0, seed=1, as_torch=True)
    for m in (uni, per):
        set_mem_cntr(m, n)
    per.sample_buffer(128)   # fills every leaf
    g = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(8):   # priorities that are not all equal
        idx = torch.randint(0, n, (65536,), device="cuda", generator=g)
        per.update_priorities(idx, torch.rand(65536, device="cuda", generator=g) * 10)
    per.check()
    return uni, per


def sample_and_update(log2, rounds=7, n=100):
    uni, per = rings(log2)
    out = {}
    for B in (1024, 4096):
        kw = dict(dtype=torch.float32, device="cuda")
        batch = (torch.empty(B, 11, **kw), torch.empty(B, 1, **kw), torch.empty(B, **kw), torch.empty(B, 11, **kw),
                 torch.empty(B, dtype=torch.uint8, device="cuda"))
        idx, w = torch.empty(B, dtype=torch.int64, device="cuda"), torch.empty(B, **kw)
        td = torch.rand(B, **kw)
        med, _ = alternate({"uniform_sample": lambda: uni.sample_buffer(B, out=batch),
                            "prioritized_sample": lambda: per.sample_buffer(B, 0.4, out=batch, idx_out=idx,
                                                                            weight_out=w),
                            "update_priorities": lambda: per.update_priorities(idx, td)}, rounds, n)
        out[B] = med
    rows = 8192 * 8

    def fill():
        set_mem_cntr(per, per.mem_cntr + rows)
        per._fill_new()
    med, _ = alternate({"fill_new_65536_rows": fill}, rounds, n)
    out["fill_new"] = med
    per.check()
    uni.close()
    per.close()
    return out


def learn(rounds=7, n=50, log2=25):
    B = 1024
    cfg = S.load_config(agent__batch_size=B)
    arms = {}
    agents = []
    for algo in ("sac1", "sac2"):
        for learner in ("fp32", "tcgen05"):
            for prioritized in (False, True):
                uni, per = rings(log2)
                (per if not prioritized else uni).close()
                torch.manual_seed(0)
                a = ContinuousAgent(cfg, None, (11,), _env_stub(), device=0, memory=per if prioritized else uni,
                                    learner_precision=learner, algorithm=algo, prioritized=prioritized)
                agents.append(a)
                arms[f"{algo}_{learner}_{'prioritized' if prioritized else 'uniform'}"] = a.learn
    med, _ = alternate(arms, rounds, n)
    for a in agents:
        a.memory.close()
    return med


def loop(iters=200):
    import train_sac
    base = ["--envs", "8192", "--iters", str(iters), "--warmup-iters", "20", "--log-every", "0", "--experiment", "6",
            "--policy-precision", "tcgen05", "--learner-precision", "tcgen05", "--collect-steps", "8",
            "--updates-per-iter", "8", "--buffer", "1000000"]
    out = {}
    for algo in ("sac1", "sac2"):
        for name, extra in (("uniform", []), ("prioritized", ["--prioritized"])):
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                summary = train_sac.main(base + ["--algorithm", algo] + extra)
            out[f"{algo}_{name}"] = summary
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="per_eval.json")
    ap.add_argument("--skip-loop", action="store_true")
    args = ap.parse_args()
    res = {"card": card()}
    res["sample_update_ms"] = {f"2^{k}": sample_and_update(k) for k in (20, 25)}
    res["learn_ms_batch1024_ring2^25"] = learn()
    if not args.skip_loop:
        res["train_sac_loop"] = loop()
    m = res["learn_ms_batch1024_ring2^25"]
    res["v2_fused_prioritized_over_uniform"] = m["sac2_tcgen05_prioritized"] / m["sac2_tcgen05_uniform"]
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
