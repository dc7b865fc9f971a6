#!/usr/bin/env python
"""The fused tcgen05 learner (ContinuousAgent(learner_precision="tcgen05"), csrc/learner.cu) against the captured fp32
update graph on one GPU.

    python profiles/learner_eval.py --out learner_eval.json [--driver] [--learning]

Per update: B = 256, 1024 and 4096, two agents from the same weights and batch, the fp32 graph replay and the two
fused kernels timed with CUDA events over 50 updates each, alternating between the two learners for 7 rounds after
warm-up; medians are reported.  The batch and the weights are a few MB, so both learners run from L2.  Before the
timing, one update of the fused learner on that batch is checked against the bf16 emulation of
tests/test_gpu_learner.py (the test's tolerance).

--driver times examples/train_sac.py at 8192 envs with --policy-precision tcgen05 --collect-steps 8
--updates-per-iter 8 under both learners (ms per env step).  --learning runs the r02f learning run (experiment 6,
8192 envs, reference hyper-parameters, 2 updates per iteration, a 33,554,432-slot ring, 40,000 iterations) with
--learner-precision tcgen05 into --artefacts (the reference's experiment tree) and reports the best interval score
and how many episodes reached the goal.  The card's
name and power limit are read in the same run.  One JSON document, printed and written to --out.
"""
import argparse
import csv
import glob
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from test_gpu_learner import _agent, _params, _random_batch, emulate_update, TRAINED  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:  # reported, not guessed
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def check_against_emulation(agent, batch):
    """worst |grad - emulation| / max|grad| over the 26 tensors after one update."""
    L = agent.learner
    P = _params(L)
    grads, losses = emulate_update(P, batch["state"], batch["action"], batch["reward"], batch["new_state"],
                                   batch["done"], batch["eps"], L.gamma, L.scale)
    got = agent.learn_from(batch["state"], batch["action"], batch["reward"], batch["new_state"],
                           batch["done"].to(torch.uint8), eps=batch["eps"])
    torch.cuda.synchronize()
    worst = 0.0
    for n in TRAINED:
        for k, p in getattr(L, n).named_parameters():
            ref = grads[n][k]
            worst = max(worst, (p.grad - ref).abs().max().item() / max(ref.abs().max().item(), 1e-12))
    loss_err = ((torch.stack([x.detach() for x in got]) - losses).abs() / losses.abs().clamp_min(1e-6)).max().item()
    return worst, loss_err


def per_update(B, rounds=7, n=50):
    agents = {lp: _agent(B, learner_precision=lp, seed=B) for lp in ("fp32", "tcgen05")}
    agents["tcgen05"].load_state_dict(agents["fp32"].state_dict())
    b = _random_batch(B, B)
    grad_err, loss_err = check_against_emulation(agents["tcgen05"], b)
    for a in agents.values():
        for dst, src in zip(a._batch, (b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8))):
            dst.copy_(src.reshape(dst.shape))
        a._eps.copy_(b["eps"])
        for _ in range(10):   # warm-up (the fp32 learner captures its graph here)
            a._run_update()
    torch.cuda.synchronize()
    times = {lp: [] for lp in agents}
    for _ in range(rounds):
        for lp, a in agents.items():
            times[lp].append(timed(a._run_update, n))
    med = {lp: statistics.median(t) for lp, t in times.items()}
    for a in agents.values():
        a.memory.close()
    return {"batch": B, "ms_per_update_fp32_graph": med["fp32"], "ms_per_update_tcgen05": med["tcgen05"],
            "speedup": med["fp32"] / med["tcgen05"], "all_ms": times,
            "tcgen05_vs_emulation_worst_grad_err": grad_err, "tcgen05_vs_emulation_worst_loss_rel_err": loss_err}


def driver(learner):
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train_sac.py"), "--envs", "8192", "--iters", "300",
           "--warmup-iters", "20", "--experiment", "6", "--policy-precision", "tcgen05", "--collect-steps", "8",
           "--updates-per-iter", "8", "--learner-precision", learner]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        return {"learner_precision": learner, "error": (r.stderr or r.stdout)[-2000:]}
    d = json.loads(lines[-1])
    return {"learner_precision": learner, "ms_per_env_step": d["ms_per_iter"] / 8, "summary": d}


def learning(root):
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train_sac.py"), "--envs", "8192", "--iters", "40000",
           "--warmup-iters", "20", "--updates-per-iter", "2", "--experiment", "6", "--buffer", "33554432",
           "--log-every", "1000", "--experiments-root", root, "--learner-precision", "tcgen05"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    res = {"cmd": " ".join(["examples/train_sac.py"] + cmd[2:-4] + cmd[-2:]), "returncode": r.returncode}
    if lines:
        res["summary"] = json.loads(lines[-1])
        res["summary"]["experiment_dir"] = os.path.relpath(res["summary"]["experiment_dir"], root)
    consoles = glob.glob(os.path.join(root, "**", "console.csv"), recursive=True)
    if consoles:
        rows = list(csv.DictReader(open(consoles[0])))
        res["console_rows"] = rows
    if r.returncode != 0:
        res["error"] = r.stderr[-2000:]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--driver", action="store_true")
    ap.add_argument("--learning", action="store_true")
    ap.add_argument("--artefacts", default=None,
                    help="directory for the learning run's experiment tree (default: a new temporary directory)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "learner_eval needs the GPU"
    res = {"card": card(), "per_update": [per_update(B) for B in (256, 1024, 4096)]}
    for r in res["per_update"]:
        print(f"B={r['batch']}: fp32 graph {r['ms_per_update_fp32_graph']:.4f} ms, tcgen05 {r['ms_per_update_tcgen05']:.4f} ms "
              f"({r['speedup']:.2f}x); vs emulation {r['tcgen05_vs_emulation_worst_grad_err']:.2e}", file=sys.stderr)
    if args.driver:
        res["train_sac_8192"] = [driver(lp) for lp in ("fp32", "tcgen05")]
    if args.learning:
        res["learning_r02f_tcgen05"] = learning(args.artefacts or tempfile.mkdtemp(prefix="learner_eval_"))
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
