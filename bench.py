#!/usr/bin/env python
"""bench.py -- batched BoatEnv env-steps/s on N B200s (BASELINE.json metric) with the HBM
roofline of the step kernel and the CPU baseline timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling weak|strong]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[2]): BoatEnv experiment 6 (changing velocity, random
direction), fp32 production mode, uniform(-1,1) policy "A1" (SURVEY.md 8d) so episodes end by
rudder_broken every ~360 steps and the in-kernel auto-reset runs in steady state.
``--scaling weak`` (default): 16,777,216 envs PER GPU; ``--scaling strong``: 16,777,216 envs in
TOTAL, sharded over the ranks by ``shard_range`` (2,097,152 per GPU at N = 8).  Envs shard with no
data-path collective.

A "step" is one BoatEnv.step over every env of the rank: one action-fill launch (the policy) + one
step launch; actions are read from an [n_envs] float32 tensor (the API-faithful variant).  Before
any timing the population is PRE-ROLLED by PREROLL untimed steps so that episode ends (and the
in-kernel resets they trigger) run at their steady-state rate whatever --warmup is; the number of
episodes that finished inside the timed region is printed.  The 64-byte statistics vector is
all-reduced (NCCL) every STATS_EVERY steps and at least once inside the timed region.  Every step
streams ~2.8 GB per GPU (>> 126 MB L2) under weak scaling; under strong scaling at N = 8 a rank's
state (118 MB) fits the L2, which the config line says.

``--impl reference`` times the UNMODIFIED reference ``BoatEnv`` (environment/boat_env.py, staged
by oracle/make_ref.py into oracle/_ref so that it travels to the GPU box) on all host cores, one
process per core in the reference's own fan-out style (main.py:215-235), on bounded samples of the
same workload; if the staged copy is missing it falls back to the C port (oracle/boat_oracle.c).

``--dump-outputs DIR`` writes, after the timed steps, what the last timed step gave its caller (the policy's
actions and BoatEnv.step's obs / reward / done / term / final_obs) as DIR/<name>.npy, float32, for a fixed
seeded sample of DUMP_ENVS envs of rank 0 (all of them when it has fewer), and the sampled env ids as
DIR/env_index.npy, float64.  The inputs depend only on the arguments, so two builds run with the same
arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "batched BoatEnv env-steps/sec at 1/2/4/8 B200; % of HBM roofline"  # BASELINE.json "metric", verbatim
UNIT = "env-steps/s"
ENVS_PER_GPU = 16_777_216
EXPERIMENT = 6
SEED = 1
ALGO_BYTES_PER_STEP = 165  # SURVEY.md 8(d): fp32, K=1, exp 6: action 4 + state 56 read + 56 write + obs 44 + reward 4 + done 1
STATS_EVERY = 250          # NCCL all-reduce of the 64-byte statistics vector every M steps (and once per timed region)
PREROLL = 1000             # untimed steps before warm-up: brings the reset rate to its steady state (episodes last ~360 steps)
DUMP_ENVS = 1 << 18        # --dump-outputs: envs sampled (26 floats each: ~27 MB in all, under the 64 MB cap)
DUMP_SEED = 12345


def workload_config(n_gpus: int, envs_per_gpu: int, scaling: str = "weak", total_envs: int | None = None) -> dict:
    total = envs_per_gpu * n_gpus if total_envs is None else total_envs
    l2 = ("inputs larger than L2 (about %.1f GB streamed per step per GPU vs 126 MB L2); no flush" % (envs_per_gpu * 165 / 1e9)
          if envs_per_gpu * 165 > 4 * 126e6 else
          "per-GPU state (%.0f MB) is comparable to the 126 MB L2: consecutive launches alternate their sweep direction, "
          "part of the state is an L2 hit; outputs (obs / reward / done) stream to HBM" % (envs_per_gpu * 72 / 1e6))
    return {"workload": f"BoatEnv experiment {EXPERIMENT} (changing velocity, random direction), fp32, "
                        f"{envs_per_gpu} envs per GPU, uniform(-1,1) policy, auto-reset in steady state "
                        f"({PREROLL}-step untimed pre-roll), K=1 sub-step per launch",
            "experiment": EXPERIMENT, "envs_per_gpu": envs_per_gpu, "total_envs": total,
            "precision": "fp32", "substeps_per_launch": 1, "policy": "uniform(-1,1) Philox(seed, env, step)",
            "seed": SEED, "preroll_steps": PREROLL, "scaling": scaling,
            "sharding": f"{n_gpus} x contiguous env-id blocks, no data-path collective; statistics all-reduce every "
                        f"{STATS_EVERY} steps and once per timed region",
            "l2_policy": l2}


def hbm_peak() -> tuple[float, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(envs_per_gpu: int):
    """dram bytes per launch of the step kernel from the committed ncu --set full capture
    (profiles/step_kernel_traffic.json), if it was taken at this problem size."""
    try:
        with open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")) as f:
            d = json.load(f)
        if int(d.get("n_envs", -1)) == envs_per_gpu:
            return float(d["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, cuda_index: int, period: float = 0.01):
        super().__init__(daemon=True)
        self.period = period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            try:  # CUDA ordinals follow CUDA_VISIBLE_DEVICES, NVML's do not: go through the PCI address
                pr = torch.cuda.get_device_properties(cuda_index)
                bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self) -> dict:
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# -------------------------------------------------------------------------------------
# CPU side: the oracle port of the reference algorithm on the host cores
# -------------------------------------------------------------------------------------
def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class CpuPort:
    """The reference's per-episode CPU stepping (boat_env.py:67-126, wind.py:26-99) as restated
    in oracle/boat_oracle.c, pthreads over independent envs, same experiment / policy /
    auto-reset as the GPU workload."""

    def __init__(self, threads: int):
        import numpy as np
        from oracle import oracle as O
        import sac_agent_b200 as S
        self.np, self.O = np, O
        self.threads = threads
        self.params = O.params_from_config(S.load_config(base_settings__experiment=EXPERIMENT))
        self.rng = np.random.default_rng(SEED)

    def sample(self, n_envs: int, t_steps: int) -> tuple[int, float]:
        np = self.np
        episodes = max(8, t_steps // 20 + 2)
        actions = self.rng.uniform(-1, 1, size=(t_steps, n_envs)).astype(np.float32).astype(np.float64)
        s_y = self.rng.integers(-640, 640, size=(episodes, n_envs)).astype(np.int32)
        knots = self.rng.random((episodes, n_envs, 2, 8))
        t0 = time.perf_counter()
        out = self.O.rollout(self.params, actions, s_y, knots, auto_reset=True, want_obs=False,
                             n_threads=self.threads)
        return int(out["steps"]), time.perf_counter() - t0


def port_baseline(target_seconds: float = 10.0) -> dict:
    """The C port of the reference algorithm (oracle/boat_oracle.c) on all cores and on one core."""
    cores = host_cores()
    port = CpuPort(cores)
    t_steps = 1000
    steps, dt = port.sample(16 * cores, t_steps)          # calibration, also warms the threads
    rate = steps / dt
    n_envs = int(max(16 * cores, min(rate * target_seconds / t_steps, 4_000_000 // t_steps * 16)))
    n_envs = (n_envs + 15) // 16 * 16
    reps = max(1, min(4, int(round(target_seconds * rate / (n_envs * t_steps)))))  # memory-bounded chunks
    steps = dt = 0.0
    for _ in range(reps):
        s_, d_ = port.sample(n_envs, t_steps)
        steps += s_
        dt += d_
    one = CpuPort(1)                                       # the same port on ONE core: a ~2 s sample
    n1 = max(16, int(rate / cores * 2.0 / t_steps))
    s1, d1 = one.sample(n1, t_steps)
    return {"value": steps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{reps} x {n_envs} envs x {t_steps} steps, experiment {EXPERIMENT}, uniform(-1,1) actions, "
                      f"auto-reset, oracle/boat_oracle.c with {cores} pthreads ({dt:.1f} s)",
            "value_1core": s1 / d1, "sample_1core": f"{n1} envs x {t_steps} steps on one thread ({d1:.1f} s)"}


def reference_available() -> bool:
    try:
        from oracle import ref_bench
        return ref_bench.available()
    except Exception:
        return False


def cpu_baseline_leg(target_seconds: float = 10.0) -> dict:
    """cpu_baseline of the bench line.  kind "reference": the UNMODIFIED reference BoatEnv (Python; BASELINE.md
    section 3) on P = all host cores, one process and one env per core, and on one core; the C port's figures
    ride along under "port".  Without the staged reference (oracle/_ref) the port is the baseline."""
    port = port_baseline(target_seconds)
    if not reference_available():
        return port
    from oracle import ref_bench
    cores = host_cores()
    allc = ref_bench.measure(cores, target_seconds, EXPERIMENT, SEED)
    one = ref_bench.measure(1, 4.0, EXPERIMENT, SEED)
    return {"value": allc["value"], "unit": UNIT, "cores": cores, "kind": "reference",
            "sample": f"unmodified reference BoatEnv (environment/boat_env.py under oracle/ref_shim.py stubs), experiment "
                      f"{EXPERIMENT}, {cores} processes x 1 env, float32-representable uniform(-1,1) actions as float64, resets included: "
                      f"{allc['steps']} env-steps in {allc['seconds']:.1f} s ({allc['episodes']} episodes)",
            "value_1core": one["value"],
            "sample_1core": f"1 process: {one['steps']} env-steps in {one['seconds']:.1f} s",
            # the names BASELINE.md section 3 announces
            "cpu_steps_per_s_1core": one["value"], "cpu_steps_per_s_allcores": allc["value"], "cpu_cores": cores,
            "port": port}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    total = max(1, args.steps + args.warmup)
    budget = args.ref_budget_s / total                     # seconds per bench "step"
    if reference_available() and not args.ref_port:
        from oracle import ref_bench
        pool = ref_bench.ReferencePool(cores, EXPERIMENT, SEED)
        n, wall, _ = pool.run(1500)                        # imports, first episode, calibration
        per_proc = max(200, int(n / cores / wall * budget))
        for _ in range(args.warmup):
            pool.run(per_proc)
        done_steps, elapsed, episodes = 0, 0.0, 0
        for _ in range(args.steps):
            n, wall, eps = pool.run(per_proc)
            done_steps += n
            elapsed += wall
            episodes += eps
        pool.close()
        kind = "reference"
        sample = (f"each step = {cores} processes x 1 env x {per_proc} env-steps of the UNMODIFIED reference BoatEnv "
                  f"(environment/boat_env.py, staged by oracle/make_ref.py), experiment {EXPERIMENT}, float32-representable uniform(-1,1) "
                  f"actions as float64, resets included ({episodes} episodes in the timed steps)")
        ran = {"implementation": "reference BoatEnv (Python, unmodified)", "processes": cores, "envs": cores,
               "env_steps_per_process_per_step": per_proc, "experiment": EXPERIMENT, "precision": "fp64 (numpy scalars)"}
    else:
        port = CpuPort(cores)
        t_steps = 500
        steps, dt = port.sample(16 * cores, t_steps)
        rate = steps / dt
        n_envs = int(max(cores, min(rate * budget / t_steps, 65536)))
        for _ in range(args.warmup):
            port.sample(n_envs, t_steps)
        done_steps, elapsed = 0, 0.0
        for _ in range(args.steps):
            s, dt = port.sample(n_envs, t_steps)
            done_steps += s
            elapsed += dt
        kind = "port"
        sample = (f"each step = {n_envs} envs x {t_steps} env-steps of experiment {EXPERIMENT}, uniform(-1,1) actions, "
                  f"auto-reset; oracle/boat_oracle.c (C port of boat_env.py/wind.py), {cores} pthreads")
        ran = {"implementation": "oracle/boat_oracle.c (C port)", "threads": cores, "envs": n_envs,
               "env_steps_per_env_per_step": t_steps, "experiment": EXPERIMENT, "precision": "fp64"}
    value = done_steps / elapsed if elapsed > 0 else 0.0
    cfg = workload_config(args.gpus, args.envs_per_gpu, args.scaling)   # the GPU arm's workload ...
    cfg["reference_arm_ran"] = ran                                      # ... and the bounded sample of it this arm really ran
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / max(1, args.steps),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------
# GPU side
# -------------------------------------------------------------------------------------
def run_ours(args) -> None:
    import torch
    import torch.distributed as dist
    import sac_agent_b200 as S

    rank, local_rank, world = S.sharding.dist_info()
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = S.sharding.bind_to_gpu_numa_node(local_rank) if world > 1 else []
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = S.lib()

    if args.scaling == "strong":   # 16,777,216 envs in TOTAL (SURVEY.md 8d config 3), contiguous shards
        total_envs = args.total_envs
        offset, n_local = S.sharding.shard_range(total_envs, rank, world)
    else:                           # 16,777,216 envs PER GPU
        n_local = args.envs_per_gpu
        total_envs = n_local * world
        offset = rank * n_local
    cfg = S.load_config(base_settings__experiment=EXPERIMENT)
    env = S.BatchedBoatEnv(cfg, n_local, seed=SEED, precision="fp32", device=local_rank,
                           env_id_offset=offset, auto_reset=True)
    env.reset()
    actions = torch.empty(n_local, dtype=torch.float32, device=dev)
    stats = torch.zeros(8, dtype=torch.float64, device=dev)
    n_allreduce = [0]

    def reduce_stats():
        """The only exchange of the path: all-reduce of the 64-byte statistics vector (SURVEY.md 8e)."""
        env._L.boatenv_reduce_counters(env._h, stats.data_ptr(), env._stream())
        if world > 1:
            dist.all_reduce(stats)
        n_allreduce[0] += 1

    def one_step(t, ev=None, force_stats=False):
        env.uniform_actions(t, args.action_scale, out=actions)       # the policy (1 launch)
        if ev is not None:
            ev[0].record()
        out = env.step(actions)                         # BoatEnv.step for every env (1 launch)
        if ev is not None:
            ev[1].record()
        if (t + 1) % STATS_EVERY == 0 or force_stats:   # occasional statistics all-reduce
            reduce_stats()
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # everything slow on the host (NVML initialisation, event creation) happens BEFORE the warm-up, so that the GPU
    # goes from the last warm-up step into the timed region without idling (a ~100 ms idle gap lets the clocks drop
    # and made a 20-step timed region read 2-3 % slower than a 1000-step one)
    kernel_events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                     for _ in range(args.steps)]
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank)
    t = 0
    for _ in range(PREROLL):                            # untimed pre-roll to the steady-state reset rate
        one_step(t)
        t += 1
    reduce_stats()
    episodes_before_warmup = float(stats[5].item())
    sampler.start()
    for _ in range(args.warmup):                        # W untimed warm-up steps, straight into the timed region
        one_step(t)
        t += 1
    barrier()
    launches0 = lib.boatenv_kernel_launches()
    n_allreduce[0] = 0
    start.record()
    for k in range(args.steps):
        # the statistics all-reduce fires inside every timed region, however short (here: at its middle step)
        last = one_step(t, kernel_events[k], force_stats=(k == args.steps // 2))
        t += 1
    end.record()
    barrier()
    launches = lib.boatenv_kernel_launches() - launches0
    clocks = sampler.stop()
    allreduces_timed = n_allreduce[0]
    if args.dump_outputs and rank == 0:
        obs, reward, done, info = last
        dump_outputs(args.dump_outputs, {"action": actions, "obs": obs, "reward": reward, "done": done,
                                         "term": info["term"], "final_obs": info["final_obs"]})
    reduce_stats()
    # episodes that ended in warm-up + timed steps, scaled to the timed steps (the rate is steady after the pre-roll;
    # counting exactly would need a host read-back between warm-up and timed region, i.e. the idle gap avoided above)
    episodes_timed = (float(stats[5].item()) - episodes_before_warmup) * args.steps / (args.steps + args.warmup)
    elapsed_ms = start.elapsed_time(end)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kernel_events) / max(1, args.steps)
    tmax = torch.tensor([elapsed_ms, kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    elapsed_ms, kernel_ms = float(tmax[0]), float(tmax[1])
    value = total_envs * args.steps / (elapsed_ms * 1e-3)

    # ---- e2e: the same metric through the public API with HOST buffers -------------------
    if args.no_e2e:  # profiling runs (ncu): the device-timed part only
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                              "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "kernel_ms": kernel_ms,
                              "gpu_launches": int(launches), "clocks": clocks,
                              "episodes_finished_in_timed_region": episodes_timed, "note": "--no-e2e profiling run"}),
                  flush=True)
        env.close()
        if world > 1:
            dist.destroy_process_group()
        return
    e2e_steps = max(3, min(args.e2e_steps, args.steps))
    act_h = torch.empty(n_local, dtype=torch.float32).pin_memory()
    obs_h = torch.empty((n_local, 11), dtype=torch.float32).pin_memory()
    rew_h = torch.empty(n_local, dtype=torch.float32).pin_memory()
    done_h = torch.empty(n_local, dtype=torch.uint8).pin_memory()
    act_h.copy_(env.uniform_actions(t, 1.0))
    for _ in range(2):
        env.step_host(act_h, obs_h, rew_h, done_h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        env.step_host(act_h, obs_h, rew_h, done_h)      # blocks until results are in host memory
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = total_envs * e2e_steps / float(te[0])
    h2d = act_h.numel() * act_h.element_size()
    d2h = sum(x.numel() * x.element_size() for x in (obs_h, rew_h, done_h))

    # ---- second e2e line: K = 8 sub-steps per host round trip (boatenv_step_k_host) ----------
    e2e_k = None
    if args.e2e_k > 1:
        K = args.e2e_k
        act_k = torch.empty((K, n_local), dtype=torch.float32).pin_memory()
        for q in range(K):
            act_k[q].copy_(env.uniform_actions(t + q, 1.0))
        for _ in range(2):
            env.step_k_host(act_k, K, obs_h, rew_h, done_h)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            env.step_k_host(act_k, K, obs_h, rew_h, done_h)
        torch.cuda.synchronize()
        tk = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tk, op=dist.ReduceOp.MAX)
        # executed sub-steps: an env that ends inside a window stops there (about K/360 of the envs per window)
        e2e_k = {"value": total_envs * K * e2e_steps / float(tk[0]), "unit": UNIT, "substeps_per_call": K,
                 "h2d_bytes_per_step": act_k.numel() * act_k.element_size(), "d2h_bytes_per_step": d2h,
                 "steps": e2e_steps, "api": "BatchedBoatEnv.step_k_host (boatenv_step_k_host): actions [K][N] in, one "
                                            "observation / summed reward / done per env out",
                 "note": "upper bound by < K/360: windows in which an episode ends execute fewer than K sub-steps"}
    counters = S.all_reduce_counters(env.counters_tensor())

    # ---- configs[3]: toy_car / toy_parachute, 1 M envs each, fp32 (rank 0, device-timed) ---------
    toys = None
    if rank == 0 and not args.no_toys:
        toys = toy_timings(S, torch, local_rank)

    if rank == 0:
        peak, peak_src = hbm_peak()
        achieved = ALGO_BYTES_PER_STEP * n_local / (kernel_ms * 1e-3) / 1e9
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(world, n_local, args.scaling, total_envs),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": ncu_traffic(n_local),
                             "kernel": "boat_step_kernel<float, WIND_BOTH>", "kernel_ms": kernel_ms,
                             "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_STEP,
                             "algorithmic_bytes_per_launch": ALGO_BYTES_PER_STEP * n_local, "peak_source": peak_src,
                             "whole_step_frac": ALGO_BYTES_PER_STEP * n_local / (elapsed_ms / args.steps * 1e-3) / 1e9 / peak},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": e2e_steps, "api": "BatchedBoatEnv.step_host (boatenv_step_host_stream, pinned host buffers)",
                        "rank0_cpu_affinity": len(numa_cpus) or None},
                "e2e_k": e2e_k,
                "gpu_launches": int(launches), "clocks": clocks,
                "episodes_finished_in_timed_region": episodes_timed,
                "stats_allreduces_in_timed_region": allreduces_timed,
                "episodes_finished": counters["episodes"], "mean_episode_return": counters["return_mean"],
                "toys": toys}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_leg() if world == 1 else None
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """--dump-outputs: the rows of a fixed seeded env sample of every output tensor, as float32 .npy files."""
    import numpy as np
    import torch
    n = outputs["obs"].shape[0]
    idx = np.arange(n)
    if n > DUMP_ENVS:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=DUMP_ENVS, replace=False))
    rows = torch.from_numpy(idx).to(outputs["obs"].device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    for name, x in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), x.index_select(0, rows).float().cpu().numpy())


def toy_timings(S, torch, device: int) -> dict:
    """BASELINE.json configs[3]: toy_car and toy_parachute, 1,048,576 envs each, fp32, on one B200.  Device-timed
    (CUDA events), whole scripts: 5001 iterations of toy_car.py:19-32, 2654 of toy_parachute.py:16-40."""
    out = {}
    n = 1 << 20
    for kind, iters in (("car", 5001), ("parachute", 2654)):
        try:
            toy = (S.ToyCar if kind == "car" else S.ToyParachute)(n, jitter=0.1, seed=1, precision="fp32", device=device)
            toy.reset()
            toy.step(iters)                               # warm-up
            toy.reset()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            toy.step(iters)
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b)
            out[kind] = {"envs": n, "iterations": iters, "ms": ms, "env_iterations_per_s": n * iters / (ms * 1e-3),
                         "precision": "fp32"}
            toy.close()
        except Exception as e:  # the toys are a secondary config: never lose the headline line over them
            out[kind] = {"error": repr(e)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="device-timed part only (for ncu runs)")
    ap.add_argument("--action-scale", type=float, default=1.0, help="experiments only: scale of the uniform policy")
    ap.add_argument("--ref-budget-s", type=float, default=90.0, help="--impl reference: CPU seconds for all steps together")
    ap.add_argument("--ref-port", action="store_true", help="--impl reference: time the C port even if the staged reference exists")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak")
    ap.add_argument("--total-envs", type=int, default=ENVS_PER_GPU, help="--scaling strong: envs over all GPUs")
    ap.add_argument("--e2e-k", type=int, default=8, help="sub-steps per host round trip of the second e2e line (0: skip)")
    ap.add_argument("--no-toys", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (a fixed sample of the envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
