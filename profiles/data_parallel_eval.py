#!/usr/bin/env python
"""Data-parallel SAC updates (ContinuousAgent(data_parallel=...)) against today's single-agent update.

    python profiles/data_parallel_eval.py --out data_parallel_eval.json

One GPU, world 1: for both learners (the captured fp32 graph and the fused tcgen05 kernels) at B = 256, 1024 and 4096,
a plain agent and a data-parallel agent on a one-rank NCCL group start from the same weights and batch.  The
data-parallel update is the split one: gradients (fp32: graph A; tcgen05: boatagent_sac_gradients), the all-reduce of
the flat gradient + loss buffer, DeviceAdam (fp32: graph B).  Both agents' losses and training tensors are compared
bit for bit after their first update and again after the timing (both made the same updates on the same batch).
Timing: CUDA events over 50 updates, alternating between the two agents for 7 rounds after 10 warm-up updates;
medians.  The batch and the weights are a few MB, so both run from L2.

With at least two visible GPUs, it also runs itself under torchrun (NCCL) at world 2 / 4 / 8 (as many as there are
GPUs) and reports rank 0's median time per update and, separately, of the all-reduce alone; with one GPU these rows
are "not measured".  The card's name and power limit are read in the same run.  One JSON document, printed and
written to --out.
"""
import argparse
import json
import os
import socket
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from learner_eval import card, timed  # noqa: E402
from test_gpu_learner import _agent, _random_batch  # noqa: E402

LEARNERS = ("fp32", "tcgen05")
BATCHES = (256, 1024, 4096)


def _load_batch(agent, b):
    for dst, src in zip(agent._batch, (b["state"], b["action"], b["reward"], b["new_state"], b["done"].to(torch.uint8))):
        dst.copy_(src.reshape(dst.shape))
    agent._eps.copy_(b["eps"])


def _same(a, b):
    torch.cuda.synchronize()
    return all(torch.equal(x, y) for x, y in zip(a.training_tensors(), b.training_tensors())) and \
        torch.equal(torch.stack(list(a._losses)), torch.stack(list(b._losses)))


def world_1(learner, B, rounds=7, n=50):
    plain = _agent(B, learner_precision=learner, seed=B)
    dp = _agent(B, learner_precision=learner, seed=B + 1, data_parallel=True)
    dp.load_state_dict(plain.state_dict())
    b = _random_batch(B, B)
    for a in (plain, dp):
        _load_batch(a, b)
        a._run_update()
    first = _same(plain, dp)
    for a in (plain, dp):
        for _ in range(10):
            a._run_update()
    torch.cuda.synchronize()
    times = {"plain": [], "data_parallel": []}
    for _ in range(rounds):
        for k, a in (("plain", plain), ("data_parallel", dp)):
            times[k].append(timed(a._run_update, n))
    last = _same(plain, dp)
    for a in (plain, dp):
        a.memory.close()
    med = {k: statistics.median(t) for k, t in times.items()}
    return {"learner_precision": learner, "batch": B, "ms_per_update_plain": med["plain"],
            "ms_per_update_data_parallel_world_1": med["data_parallel"], "ratio": med["data_parallel"] / med["plain"],
            "bit_identical_after_first_update": first, "bit_identical_after_timing": last, "all_ms": times}


def worker(out):
    """One rank of the torchrun measurement: per learner and batch, time per data-parallel update and per all-reduce."""
    rank, local_rank, world = (int(os.environ[k]) for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rows = []
    for learner in LEARNERS:
        for B in BATCHES:
            a = _agent(B, learner_precision=learner, seed=B, data_parallel=True)
            _load_batch(a, _random_batch(B, B + rank))
            flat = a._dp[1]
            for _ in range(10):
                a._run_update()
            upd, red = [], []
            for _ in range(7):
                upd.append(timed(a._run_update, 50))
                red.append(timed(lambda: dist.all_reduce(flat), 50))
            rows.append({"learner_precision": learner, "batch": B, "world": world, "effective_batch": world * B,
                         "ms_per_update": statistics.median(upd), "ms_per_all_reduce": statistics.median(red),
                         "all_reduce_bytes": flat.numel() * 4})
            a.memory.close()
    if rank == 0:
        with open(out, "w") as f:
            json.dump(rows, f)
    dist.destroy_process_group()


def multi_gpu(tmp):
    n = torch.cuda.device_count()
    res = {}
    for world in (2, 4, 8):
        if world > n:
            res[f"world_{world}"] = f"not measured ({n} GPU{'s' if n != 1 else ''} visible)"
            continue
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        out = os.path.join(tmp, f"world_{world}.json")
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__),
                            "--worker", out], capture_output=True, text=True, timeout=1800)
        res[f"world_{world}"] = json.load(open(out)) if r.returncode == 0 else {"error": r.stderr[-2000:]}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "data_parallel_eval needs the GPU"
    if args.worker:
        return worker(args.worker)
    import tempfile
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1, device_id=torch.device("cuda", 0))
    res = {"card": card(), "world_1": [world_1(lp, B) for lp in LEARNERS for B in BATCHES]}
    dist.destroy_process_group()
    for r in res["world_1"]:
        print(f"{r['learner_precision']} B={r['batch']}: plain {r['ms_per_update_plain']:.4f} ms, data-parallel world 1 "
              f"{r['ms_per_update_data_parallel_world_1']:.4f} ms ({r['ratio']:.2f}x); bit-identical "
              f"{r['bit_identical_after_first_update'] and r['bit_identical_after_timing']}", file=sys.stderr)
    with tempfile.TemporaryDirectory() as tmp:
        res["multi_gpu_nccl"] = multi_gpu(tmp)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
