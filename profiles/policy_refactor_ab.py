#!/usr/bin/env python
"""A/B of the acting kernel (boatagent_policy_act, csrc/policy_mlp.cu) between two libboatenv builds: a baseline
library and this tree's.  Written for the change that made policy_mlp_kernel run the shared tcgen05 pass of
csrc/actor_tc.cuh instead of its own inline copy; the two builds must give the same bits at the same speed.

    python profiles/policy_refactor_ab.py --baseline-library OLD/libboatenv.so --out policy_refactor_ab.json

Each build runs in processes of its own (BOATENV_LIBRARY selects the library).
  * actions: n_actions 1, 2, 4, 8 x obs_dim 5, 11, 16 x (given eps, Philox draws) x n = 1, 127, 128, 70,001 and
    1,048,576 envs, from seeded inputs (random actor, standard-normal observations and eps, a 64-bit seed, a step
    counter above 2^32).  Every output is compared bit for bit.
  * time: the kernel at 65,536 and 1,048,576 envs (n_actions 1, obs_dim 11, Philox draws), CUDA events around
    back-to-back launches called straight through ctypes (the inputs stay in L2 between launches).  The builds
    alternate over --reps processes each; per build and size the median and the spread (max - min) of the
    processes' medians are reported.  The branch counts as not slower when its median exceeds the baseline's by no
    more than the larger spread.
  * bench: `bench.py --dump-outputs` with the same arguments under each build; every dumped array compared bit for
    bit (the step path and the policy's draw at bench scale).
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

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = (1, 127, 128, 70001, 1048576)
ACTIONS = (1, 2, 4, 8)
OBS_DIMS = (5, 11, 16)
SEED = 0x9E3779B97F4A7C15
STEP = (1 << 33) + 7
TIME_CALLS = {65536: 2000, 1048576: 200}
BENCH_ARGS = ["--gpus", "1", "--steps", "20", "--warmup", "5", "--no-e2e", "--no-toys", "--no-cpu-baseline"]


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:  # reported, not guessed
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def policy(na, obs_dim):
    import torch
    from sac_agent_b200.networks import ActorNetwork, TensorCorePolicy
    torch.manual_seed(100 * na + obs_dim)
    actor = ActorNetwork(None, (obs_dim,), max_action=[0.5 + 0.25 * a for a in range(na)], n_actions=na).cuda()
    return TensorCorePolicy(actor, seed=SEED)


def worker_actions(dump):
    """Every case's actions -> dump/<case>.npy."""
    import torch
    g = torch.Generator().manual_seed(7)
    n_max = max(SIZES)
    obs_all = {d: torch.randn(n_max, d, generator=g).cuda() for d in OBS_DIMS}
    eps_all = {na: torch.randn(n_max, na, generator=g).cuda() for na in ACTIONS}
    for na in ACTIONS:
        for d in OBS_DIMS:
            pol = policy(na, d)
            for draw in ("eps", "philox"):
                for n in SIZES:
                    pol.steps = STEP
                    out = pol.act(obs_all[d][:n], eps_all[na][:n] if draw == "eps" else None)
                    np.save(os.path.join(dump, f"na{na}_obs{d}_{draw}_n{n}.npy"), out.cpu().numpy())


def worker_time():
    """Median ms per call of each timed size over five windows of back-to-back launches."""
    import torch
    from sac_agent_b200 import _lib
    L = _lib.lib()
    pol = policy(1, 11)
    stream = torch.cuda.current_stream().cuda_stream
    res = {}
    for n, calls in TIME_CALLS.items():
        obs = torch.rand(n, 11, device="cuda")
        out = torch.empty(n, 1, device="cuda")
        args = (pol.blob.data_ptr(), obs.data_ptr(), None, pol.actor.max_action.data_ptr(), SEED, STEP, n, 11, 1,
                out.data_ptr(), stream)
        for _ in range(50):
            _lib.check(L.boatagent_policy_act(*args), "boatagent_policy_act")
        windows = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(calls):
                L.boatagent_policy_act(*args)
            b.record()
            torch.cuda.synchronize()
            windows.append(a.elapsed_time(b) / calls)
        _lib.check(L.boatagent_policy_act(*args), "boatagent_policy_act")
        res[str(n)] = {"ms": statistics.median(windows), "windows_ms": windows}
    return res


def run(lib, argv):
    env = dict(os.environ)
    env["BOATENV_LIBRARY"] = os.path.abspath(lib)
    return subprocess.run([sys.executable, *argv], env=env, capture_output=True, text=True, check=True, cwd=ROOT).stdout


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def compare_dirs(da, db):
    names = sorted(f for f in os.listdir(da) if f.endswith(".npy"))
    rows = []
    for f in names:
        a, b = np.load(os.path.join(da, f)), np.load(os.path.join(db, f))
        row = {"case": f[:-4], "identical": same_bits(a, b)}
        if not row["identical"] and a.shape == b.shape:
            diff = a.astype(np.float64) != b.astype(np.float64)
            row["differing"] = int(diff.sum())
            row["max_abs_diff"] = float(np.nanmax(np.abs(a.astype(np.float64) - b.astype(np.float64))))
        rows.append(row)
    return names == sorted(f for f in os.listdir(db) if f.endswith(".npy")), rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-library", help="the build to compare against")
    ap.add_argument("--library", default=None, help="this tree's build (default: the package's libboatenv.so)")
    ap.add_argument("--reps", type=int, default=7, help="timing processes per build (alternating)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", choices=["actions", "time"], help="(internal) one build's part, in its own process")
    ap.add_argument("--dump", default=None, help="(internal) where --worker actions writes")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "policy_refactor_ab needs a GPU"
    torch.cuda.set_device(0)
    if args.worker == "actions":
        worker_actions(args.dump)
        return
    if args.worker == "time":
        print(json.dumps(worker_time()))
        return

    import sac_agent_b200 as S
    builds = {"baseline": args.baseline_library, "branch": args.library or S.library_path()}
    me = os.path.abspath(__file__)
    doc = {"card": card(), "libraries": {k: os.path.relpath(os.path.abspath(v), ROOT) for k, v in builds.items()}}
    tmp = tempfile.mkdtemp(prefix="policy_ab_")
    try:
        dirs = {k: os.path.join(tmp, "actions_" + k) for k in builds}
        for k, lib in builds.items():
            os.makedirs(dirs[k])
            run(lib, [me, "--worker", "actions", "--dump", dirs[k]])
        same_cases, rows = compare_dirs(dirs["baseline"], dirs["branch"])
        doc["actions"] = {"cases": len(rows), "identical": sum(r["identical"] for r in rows),
                          "same_case_list": same_cases, "mismatches": [r for r in rows if not r["identical"]]}
        print(json.dumps({"actions": {k: v for k, v in doc["actions"].items() if k != "mismatches"}}), flush=True)

        samples = {k: [] for k in builds}
        for _ in range(args.reps):
            for k, lib in builds.items():
                samples[k].append(json.loads(run(lib, [me, "--worker", "time"]).strip().splitlines()[-1]))
        timing = {}
        for n in TIME_CALLS:
            t = {}
            for k in builds:
                ms = [s[str(n)]["ms"] for s in samples[k]]
                t[k] = {"median_ms": statistics.median(ms), "spread_ms": max(ms) - min(ms), "process_medians_ms": ms}
            t["branch_minus_baseline_ms"] = t["branch"]["median_ms"] - t["baseline"]["median_ms"]
            t["not_slower"] = t["branch_minus_baseline_ms"] <= max(t["baseline"]["spread_ms"], t["branch"]["spread_ms"])
            timing[str(n)] = t
            print(json.dumps({"envs": n, "baseline_ms": t["baseline"]["median_ms"], "branch_ms": t["branch"]["median_ms"],
                              "not_slower": t["not_slower"]}), flush=True)
        doc["time"] = {"n_actions": 1, "obs_dim": 11, "calls_per_window": {str(k): v for k, v in TIME_CALLS.items()},
                       "sizes": timing}

        bdirs = {k: os.path.join(tmp, "bench_" + k) for k in builds}
        for k, lib in builds.items():
            run(lib, [os.path.join(ROOT, "bench.py"), *BENCH_ARGS, "--dump-outputs", bdirs[k]])
        same_files, rows = compare_dirs(bdirs["baseline"], bdirs["branch"])
        doc["bench_dump"] = {"args": BENCH_ARGS, "arrays": [r["case"] for r in rows], "same_file_list": same_files,
                             "identical": all(r["identical"] for r in rows) and same_files,
                             "mismatches": [r for r in rows if not r["identical"]]}
        print(json.dumps({"bench_dump_identical": doc["bench_dump"]["identical"]}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
