#!/usr/bin/env python
"""What recording envs costs on one GPU (DeviceRecorder against no recorder and against BatchedRecorder).

    python profiles/record_overhead.py --out record_overhead.json

* the record kernel per launch at M = 1, 64, 1024 recorded envs (65,536-env population): device time of 200
  launches replayed from one CUDA graph, and the eager cost of one ``capture()`` back to back (launch + event);
* ms per iteration of the examples/train_sac.py loop (graphed policy -> fused step + store -> learn, experiment 5,
  fp32) at 65,536 and 1,048,576 envs with M = 64: no recorder, DeviceRecorder (flushes every 50 iterations timed
  apart, on the host clock, since a flush ends in a synchronise), BatchedRecorder;
* bench.py's step (a fill of uniform(-1, 1) actions, then env.step) at 16,777,216 envs (experiment 6) with and
  without a capture after every step, M = 64 and 1024.

Loop times are CUDA events around whole segments; variants alternate over the repetitions and the median is kept.
The card's name and power limit are read in the same run.  One JSON document, printed and written to --out.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import sac_agent_b200 as S  # noqa: E402
from sac_agent_b200 import _lib  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:  # reported, not guessed
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def seg_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def ids_for(env, m):
    """m ids spread over the whole population (first block, the middle, the tail)."""
    n = env.n_envs
    return sorted({int(round(k * (n - 1) / max(m - 1, 1))) for k in range(m)})[:m]


def kernel_cases(tmp):
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), 65536, seed=0, precision="fp32", device=0)
    env.reset()
    a = env.uniform_actions(0, 1.0)
    env.step(a)
    out = {}
    for m in (1, 64, 1024):
        rec = S.DeviceRecorder(env, ids_for(env, m), os.path.join(tmp, f"k{m}"), capacity=256)
        launches = 200
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            env.record_rows(rec._local, rec._ring, 0, a, env.reward, env.term)   # warm-up outside the capture
            torch.cuda.synchronize()
            with torch.cuda.graph(g, stream=s):
                for r in range(launches):
                    env.record_rows(rec._local, rec._ring, r, a, env.reward, env.term)
        torch.cuda.current_stream().wait_stream(s)
        graph_us = statistics.median(1e3 * seg_ms(g.replay, 20) / (20 * launches) for _ in range(5))
        eager = []
        for _ in range(5):
            eager.append(1e3 * seg_ms(lambda: rec.capture(a), 200) / 200)
            rec.flush()
        out[str(m)] = {"graph_us_per_launch": graph_us, "eager_us_per_capture": statistics.median(eager)}
        rec.close()
    env.close()
    return out


def sac_case(n, m, tmp, iters=200, reps=3, seg=50):
    cfg = S.load_config(base_settings__experiment=5)
    env = S.BatchedBoatEnv(cfg, n, seed=0, precision="fp32", device=0, auto_reset=True)
    mem = S.ReplayBuffer(max(1_000_000, n), (11,), 1, precision="fp32", device=0, as_torch=True)
    agent = S.ContinuousAgent(cfg, None, (11,), env, device=0, memory=mem)
    obs = env.reset()
    ids = ids_for(env, m)
    state = {"a": None}

    def it():
        state["a"] = agent.choose_action_graphed(obs).squeeze(-1)
        agent.step_and_remember(env, state["a"], done_flag_mode=1)
        agent.learn()

    for _ in range(30):   # graph captures, ring filled past one batch
        it()
    torch.cuda.synchronize()
    res = {"none": [], "device": [], "device_flush_ms": [], "batched": []}
    for rep in range(reps):
        res["none"].append(seg_ms(it, iters) / iters)
        d = os.path.join(tmp, f"sac{n}_{rep}")
        rec = S.DeviceRecorder(env, [env.env_id_offset + i for i in ids], d, capacity=seg + 1)
        rec.start()
        rec.flush()
        loop_ms, flushes = 0.0, []
        for _ in range(iters // seg):
            loop_ms += seg_ms(lambda: (it(), rec.capture(state["a"])), seg)
            t = time.perf_counter()
            rec.flush()
            flushes.append(1e3 * (time.perf_counter() - t))
        rec.close()
        res["device"].append(loop_ms / (iters // seg * seg))
        res["device_flush_ms"].append(statistics.median(flushes))
        shutil.rmtree(d, ignore_errors=True)
        d = os.path.join(tmp, f"sacb{n}_{rep}")
        brec = S.BatchedRecorder(env, ids, d)

        def it_batched():
            brec.write_data_to_csv()
            it()
            brec.after_step(state["a"])

        res["batched"].append(seg_ms(it_batched, iters // 4) / (iters // 4))
        shutil.rmtree(d, ignore_errors=True)
    out = {k: statistics.median(v) for k, v in res.items()}
    out["device_overhead_pct"] = 100.0 * (out["device"] / out["none"] - 1.0)
    out["raw"] = res
    env.close()
    mem.close()
    return out


def step_case(n, tmp, iters=500, reps=5):
    """bench.py's step: fresh uniform(-1, 1) actions (one fill launch) and env.step, with and without a capture."""
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), n, seed=0, precision="fp32", device=0)
    env.reset()
    a = env.uniform_actions(0, 1.0)
    clock = [0]

    def step():
        clock[0] += 1
        env.uniform_actions(clock[0], 1.0, out=a)
        env.step(a)

    for _ in range(50):
        step()
    recs = {m: S.DeviceRecorder(env, ids_for(env, m), os.path.join(tmp, f"step{m}"), capacity=iters + 1)
            for m in (64, 1024)}
    out = {"none": [], **{f"capture_m{m}": [] for m in recs}}
    for _ in range(reps):
        out["none"].append(1e3 * seg_ms(step, iters) / iters)
        for m, rec in recs.items():
            out[f"capture_m{m}"].append(1e3 * seg_ms(lambda: (step(), rec.capture(a)), iters) / iters)
            rec.flush()
    res = {f"{k}_us_per_step": statistics.median(v) for k, v in out.items()}
    for m in recs:
        res[f"capture_m{m}_adds_us"] = res[f"capture_m{m}_us_per_step"] - res["none_us_per_step"]
        recs[m].close()
    res["raw_us"] = out
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("record_overhead.py measures on a GPU; there is none here")
    torch.cuda.set_device(0)
    tmp = tempfile.mkdtemp(prefix="record_overhead_")
    try:
        doc = {"card": card(), "recorded_envs_m": 64}
        doc["record_kernel"] = kernel_cases(tmp)
        sizes = (4096,) if args.quick else (65536, 1048576)
        doc["train_sac_ms_per_iter"] = {str(n): sac_case(n, 64, tmp) for n in sizes}
        doc["env_step_16M"] = step_case(65536 if args.quick else 16_777_216, tmp)
        base = doc["train_sac_ms_per_iter"][str(sizes[0])]
        doc["targets"] = {
            "capture_overhead_pct_at_65536_m64": base["device_overhead_pct"], "target_pct": 2.0,
            "capture_us_per_step_16M_m64": doc["env_step_16M"]["capture_m64_adds_us"],
            "capture_us_per_step_16M_m1024": doc["env_step_16M"]["capture_m1024_adds_us"], "target_us": 5.0}
        doc["kernel_launches"] = int(_lib.lib().boatenv_kernel_launches())
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    text = json.dumps(doc, indent=1)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
