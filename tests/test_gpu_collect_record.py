"""Recording inside the fused collection kernel (boatagent_collect_record, csrc/rollout.cu; TensorCorePolicy.collect /
ContinuousAgent.collect with ``recorder=``) against the only way to record before it: per-step ``act`` +
``step_store`` followed by ``DeviceRecorder.capture``.

Bit-equal is the expected outcome everywhere: the kernel writes the rows boatenv_record_rows writes, from the same
state decoded by the same function, so the recorder rings, and the CSV files written from them, are identical.
Recording changes nothing else: the replay ring, the env state and the outputs equal those of a plain collect call
(the fp64 return sums of the counters are atomics and compared with a tolerance, as in test_gpu_collect.py).

Every test but the compiler check needs a B200 and is ``@pytest.mark.gpu``."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

COUNTER_BYTES = 32 * 32 * 8   # the counter rows at the end of an export_state blob (kCounterSlots x 32 doubles)
COUNTS = ("reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken", "episodes")
RING_COLUMNS = ("s_x", "s_y", "v_x", "v_y", "s_r", "rudder_angle", "action", "reward", "term", "episode")
EINVAL, EUNSUPPORTED, ESTATE = -1, -4, -6


@pytest.fixture(scope="module")
def S():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import sac_agent_b200 as pkg
    pkg.lib()
    return pkg


def make_actor(seed):
    """A seeded default init: it breaks the rudder or leaves the track within ~70 steps (experiment 6)."""
    import torch
    from sac_agent_b200.networks import ActorNetwork
    torch.manual_seed(seed)
    return ActorNetwork(None, (11,), max_action=[1.0]).cuda()


def policy(actor, seed=7):
    from sac_agent_b200.networks import TensorCorePolicy
    return TensorCorePolicy(actor, seed=seed)


def make_env(S, exp, n, seed=3, env_id_offset=0, precision="fp32"):
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=exp), n, seed=seed, precision=precision, device=0,
                           env_id_offset=env_id_offset, auto_reset=True)
    env.reset()
    return env


def make_ring(S, size, precision="fp32"):
    return S.ReplayBuffer(size, (11,), 1, precision=precision, device=0, as_torch=True)


def per_step(env, mem, pol, steps, rec):
    """The loop the kernel fuses, recorded the way DeviceRecorder records it."""
    for _ in range(steps):
        a = pol.act(env.obs).reshape(-1)
        mem.step_store(env, a)
        rec.capture(a)


def same(x, y):
    import torch
    if x.dtype in (torch.float32, torch.int32):
        x, y = x.contiguous().view(torch.int32), y.contiguous().view(torch.int32)
    return x.shape == y.shape and torch.equal(x, y)


def ring_rows(mem):
    import torch
    n = min(mem.mem_cntr, mem.mem_size)
    return mem.gather(torch.arange(n, dtype=torch.int64, device=mem.device), as_torch=True)


def state_part(env):
    return env.state_dict()["blob"][:-COUNTER_BYTES]


def assert_same_collect(env_f, mem_f, pol_f, env_e, mem_e, pol_e):
    assert mem_f.mem_cntr == mem_e.mem_cntr
    for k, (x, y) in enumerate(zip(ring_rows(mem_f), ring_rows(mem_e))):
        assert same(x, y), ("state", "action", "reward", "new_state", "terminal")[k]
    for name in ("obs", "reward", "done", "term"):
        assert same(getattr(env_f, name), getattr(env_e, name)), name
    assert same(state_part(env_f), state_part(env_e))
    cf, ce = env_f.counters(), env_e.counters()
    for k in COUNTS:
        assert cf[k] == ce[k], k
    for k in ("return_sum", "return_sumsq"):
        assert cf[k] == pytest.approx(ce[k], rel=1e-9, abs=1e-6), k
    assert pol_f.steps == pol_e.steps


def assert_same_recorder_ring(rec_f, rec_e):
    """All ten columns of every slot, bitwise (the rows of the two recorders sit in the same slots)."""
    import torch
    torch.cuda.synchronize()
    assert rec_f._rows == rec_e._rows and rec_f._flushed == rec_e._flushed
    for k in RING_COLUMNS:
        assert same(rec_f._cols[k], rec_e._cols[k]), k


def tree(path):
    out = {}
    for d, _, files in os.walk(path):
        for f in files:
            p = os.path.join(d, f)
            out[os.path.relpath(p, path)] = open(p, "rb").read()
    return out


def assert_same_tree(a, b):
    ta, tb = tree(a), tree(b)
    assert ta and sorted(ta) == sorted(tb)
    assert all(ta[k] == tb[k] for k in ta), [k for k in ta if ta[k] != tb[k]][:5]


def edge_ids(n, rng, extra=24):
    """Tile and warp edges, the first env of the ragged last tile, n - 1, and random ids, shuffled."""
    last_tile = (n - 1) // 128 * 128
    ids = {i for i in (0, 31, 32, 127, 128, 255, 256, last_tile, last_tile + 1, n - 1) if i < n}
    ids |= {int(i) for i in rng.choice(n, extra, replace=False)}
    ids = sorted(ids)
    rng.shuffle(ids)
    return ids


# ---------------------------------------------------------------------------------------
# 1. the ring rows are the per-step recorder's; the rest is plain collect's
# ---------------------------------------------------------------------------------------
CASES = [(e, 1000) for e in range(1, 7)] + [(2, 70000), (6, 70000), (6, 4099)]


@pytest.mark.gpu
@pytest.mark.parametrize("exp,n", CASES)
def test_ring_rows_match_per_step_recorder(S, tmp_path, exp, n):
    T = 400
    actor = make_actor(seed=1)
    ids = edge_ids(n, np.random.default_rng(exp * 100_003 + n))
    env_r, env_p, env_e = make_env(S, exp, n), make_env(S, exp, n), make_env(S, exp, n)
    mem_r, mem_p, mem_e = make_ring(S, T * n), make_ring(S, T * n), make_ring(S, T * n)
    pol_r, pol_p, pol_e = policy(actor), policy(actor), policy(actor)
    rec_r = S.DeviceRecorder(env_r, ids, str(tmp_path / "r"), capacity=T)
    rec_e = S.DeviceRecorder(env_e, ids, str(tmp_path / "e"), capacity=T)
    out = pol_r.collect(env_r, mem_r, T, recorder=rec_r)
    assert out[0] is env_r.obs and out[3]["term"] is env_r.term
    assert rec_r.pending == T and pol_r.steps == T
    pol_p.collect(env_p, mem_p, T)
    per_step(env_e, mem_e, pol_e, T, rec_e)
    assert_same_recorder_ring(rec_r, rec_e)
    assert_same_collect(env_r, mem_r, pol_r, env_p, mem_p, pol_p)
    assert bool(rec_r._cols["term"].ne(0).any())   # recorded episode ends (and the resets after them)
    for x in (env_r, env_p, env_e, mem_r, mem_p, mem_e):
        x.close()


# ---------------------------------------------------------------------------------------
# 2-4. the CSV files: automatic flushes, a wrapping call, captures in between, chunks, a shard
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_csv_trees_match_per_step_recorder(S, tmp_path):
    """Capacity 256, calls of 100 steps: flushes between calls, a call that wraps the recorder ring's end, and
    per-step capture() rounds on the same recorder between collect calls."""
    n = 1000
    ids = edge_ids(n, np.random.default_rng(3), extra=6)
    actor = make_actor(seed=2)
    plan = [100, -3, 100, 100, -2, 57]           # > 0: one collect call of that many steps, < 0: per-step rounds
    for fused in (True, False):
        env, mem, pol = make_env(S, 6, n), make_ring(S, 400 * n), policy(actor)
        rec = S.DeviceRecorder(env, ids, str(tmp_path / ("fused" if fused else "step")), capacity=256)
        rec.start()
        for k in plan:
            if fused and k > 0:
                pol.collect(env, mem, k, recorder=rec)
            else:
                per_step(env, mem, pol, abs(k), rec)
        assert rec._rows == 1 + 362 and rec._flushed > 0
        rec.close()
        assert rec.episodes_finished > len(ids)
        env.close()
        mem.close()
    assert_same_tree(tmp_path / "fused", tmp_path / "step")


@pytest.mark.gpu
def test_chunked_calls_give_the_same_files(S, tmp_path):
    n = 3000
    ids = edge_ids(n, np.random.default_rng(4), extra=8)
    actor = make_actor(seed=11)
    for name, chunks in (("whole", [400]), ("chunks", [150, 250])):
        env, mem, pol = make_env(S, 6, n), make_ring(S, 400 * n), policy(actor)
        rec = S.DeviceRecorder(env, ids, str(tmp_path / name), capacity=400)
        rec.start()
        for k in chunks:
            pol.collect(env, mem, k, recorder=rec)
        rec.close()
        env.close()
        mem.close()
    assert_same_tree(tmp_path / "whole", tmp_path / "chunks")


@pytest.mark.gpu
def test_sharded_handle_names_files_by_global_id(S, tmp_path):
    n, T, off = 1500, 300, 5000
    ids = [off + 42, off, off + 1499, off + 127, off + 128]
    actor = make_actor(seed=5)
    for fused in (True, False):
        env, mem, pol = make_env(S, 6, n, env_id_offset=off), make_ring(S, T * n), policy(actor)
        rec = S.DeviceRecorder(env, ids, str(tmp_path / ("fused" if fused else "step")), capacity=T)
        rec.start()
        if fused:
            pol.collect(env, mem, T, recorder=rec)
        else:
            per_step(env, mem, pol, T, rec)
        rec.close()
        env.close()
        mem.close()
    assert_same_tree(tmp_path / "fused", tmp_path / "step")
    names = os.listdir(tmp_path / "fused" / "episodes")
    assert {int(re.match(r"env(\d+)_", x).group(1)) for x in names} == set(ids)
    assert all(f"env{g}_wind.csv" in names and f"env{g}_episode_0_data.csv" in names for g in ids)


# ---------------------------------------------------------------------------------------
# 5. many ids: the scan with M > 128; ids outside [0, n) are skipped
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_1024_ids_over_70000_envs(S, tmp_path):
    n, T = 70000, 64
    rng = np.random.default_rng(8)
    whole_tile = list(range(300 * 128, 301 * 128))
    rest = [int(i) for i in rng.choice(np.setdiff1d(np.arange(n), whole_tile), 1024 - 128, replace=False)]
    ids = whole_tile + rest
    rng.shuffle(ids)
    actor = make_actor(seed=6)
    env_r, env_e = make_env(S, 6, n), make_env(S, 6, n)
    mem_r, mem_e = make_ring(S, T * n), make_ring(S, T * n)
    pol_r, pol_e = policy(actor), policy(actor)
    rec_r = S.DeviceRecorder(env_r, ids, str(tmp_path / "r"), capacity=T)
    rec_e = S.DeviceRecorder(env_e, ids, str(tmp_path / "e"), capacity=T)
    pol_r.collect(env_r, mem_r, T, recorder=rec_r)
    per_step(env_e, mem_e, pol_e, T, rec_e)
    assert_same_recorder_ring(rec_r, rec_e)
    for x in (env_r, env_e, mem_r, mem_e):
        x.close()


@pytest.mark.gpu
def test_ids_outside_the_env_are_skipped(S, tmp_path):
    """Local ids -1 and n passed straight to the ABI: their columns keep what the ring held; the others get the
    per-step recorder's rows."""
    import torch
    from sac_agent_b200 import _lib
    n, T, cap = 1000, 20, 32
    ids = [5, -1, 999, n, 3]
    actor = make_actor(seed=3)
    env_r, env_e = make_env(S, 6, n), make_env(S, 6, n)
    mem_r, mem_e = make_ring(S, T * n), make_ring(S, T * n)
    pol_r, pol_e = policy(actor), policy(actor)
    m = len(ids)
    cols = {k: torch.full((cap, m), -7, dtype=torch.float32, device=env_r.device) for k in RING_COLUMNS[:8]}
    cols["term"] = torch.full((cap, m), 0xAB, dtype=torch.uint8, device=env_r.device)
    cols["episode"] = torch.full((cap, m), -5, dtype=torch.int32, device=env_r.device)
    init = {k: v.clone() for k, v in cols.items()}
    ring = _lib.RecordRing(**{k: v.data_ptr() for k, v in cols.items()}, capacity=cap)
    idx = torch.tensor(ids, dtype=torch.int64, device=env_r.device)
    row0 = 3 * cap + 25                          # rows 25 .. 31 and 0 .. 12: the call wraps the ring
    L = pol_r._L
    rc = L.boatagent_collect_record(env_r._h, mem_r._h, pol_r.blob.data_ptr(), pol_r.actor.max_action.data_ptr(),
                                    pol_r.seed, 0, T, 1, env_r.obs.data_ptr(), env_r.reward.data_ptr(),
                                    env_r.done.data_ptr(), env_r.term.data_ptr(), idx.data_ptr(), m,
                                    ctypes.byref(ring), row0, torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    rec_e = S.DeviceRecorder(env_e, [5, 999, 3], str(tmp_path / "e"), capacity=T)
    per_step(env_e, mem_e, pol_e, T, rec_e)
    torch.cuda.synchronize()
    slots = [(row0 + t) % cap for t in range(T)]
    untouched = [s for s in range(cap) if s not in slots]
    for k in RING_COLUMNS:
        got = cols[k]
        assert same(got[slots][:, [0, 2, 4]], rec_e._cols[k][:T]), k
        assert same(got[:, [1, 3]], init[k][:, [1, 3]]) and same(got[untouched], init[k][untouched]), k
    for x in (env_r, env_e, mem_r, mem_e):
        x.close()


# ---------------------------------------------------------------------------------------
# 6. the agent loop with learning in between
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_agent_collect_records_like_the_per_step_loop(S, tmp_path):
    import torch
    from sac_agent_b200 import ContinuousAgent
    cfg = S.load_config(base_settings__experiment=6, agent__batch_size=256)
    ids = [0, 31, 200, 511, 128]
    runs = []
    for fused in (True, False):
        torch.manual_seed(21)
        env = S.BatchedBoatEnv(cfg, 512, seed=9, precision="fp32", device=0, auto_reset=True)
        mem = make_ring(S, 30_000)
        agent = ContinuousAgent(cfg, None, (11,), env, device=0, seed=9, memory=mem, policy_precision="tcgen05")
        env.reset()
        rec = S.DeviceRecorder(env, ids, str(tmp_path / ("fused" if fused else "step")), capacity=16)
        rec.start()
        torch.manual_seed(22)
        losses = []
        for _ in range(6):
            if fused:
                agent.collect(env, 8, recorder=rec)
            else:
                for _ in range(8):
                    actions = agent.choose_action_graphed(env.obs).squeeze(-1)
                    agent.step_and_remember(env, actions)
                    rec.capture(actions)
            for _ in range(4):
                out = agent.learn()
                assert out is not None
                losses.append(torch.stack([x.clone() for x in out]))
        rec.close()
        torch.cuda.synchronize()
        weights = [p.detach().clone() for net in agent.learner.networks() for p in net.parameters()]
        runs.append((torch.stack(losses), weights, ring_rows(mem), mem.mem_cntr))
        env.close()
    (la, wa, ra, ca), (lb, wb, rb, cb) = runs
    assert ca == cb == 6 * 8 * 512
    assert same(la, lb)
    assert all(same(x, y) for x, y in zip(wa, wb))
    assert all(same(x, y) for x, y in zip(ra, rb))
    assert_same_tree(tmp_path / "fused", tmp_path / "step")


# ---------------------------------------------------------------------------------------
# 7. errors: a rejected call changes nothing
# ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_collect_record_error_codes(S, tmp_path):
    import torch
    from sac_agent_b200 import _lib
    pol = policy(make_actor(seed=1))
    L = pol._L
    st = torch.cuda.current_stream().cuda_stream
    env = make_env(S, 6, 64)
    mem = make_ring(S, 10_000)
    rec = S.DeviceRecorder(env, [0, 5, 63], str(tmp_path), capacity=8)
    idx = rec._local

    def call(e=env, m=mem, ids=True, n_ids=3, ring=True, row=0, steps=4, cols=None, cap=8):
        if ring:
            ptrs = {k: v.data_ptr() for k, v in rec._cols.items()} | (cols or {})
            r = ctypes.byref(_lib.RecordRing(**ptrs, capacity=cap))
        else:
            r = None
        return L.boatagent_collect_record(e._h, m._h, pol.blob.data_ptr(), pol.actor.max_action.data_ptr(), 7, 0,
                                          steps, 1, e.obs.data_ptr(), e.reward.data_ptr(), e.done.data_ptr(),
                                          e.term.data_ptr(), idx.data_ptr() if ids else None, n_ids, r, row, st)

    torch.cuda.synchronize()
    before = state_part(env).clone(), env.obs.clone(), rec._buf.clone()
    assert call(ids=False) == EINVAL
    assert call(ring=False) == EINVAL
    for k in RING_COLUMNS:
        assert call(cols={k: None}) == EINVAL, k
    assert call(n_ids=0) == EINVAL
    assert call(n_ids=2 ** 31) == EINVAL
    assert call(cap=0) == EINVAL
    assert call(row=-1) == EINVAL
    assert call(steps=9) == EINVAL               # steps > capacity
    env64 = make_env(S, 6, 64, precision="fp64")
    assert call(e=env64) == EUNSUPPORTED
    fresh = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), 64, precision="fp32", device=0)
    assert call(e=fresh) == ESTATE
    assert call(steps=0) == EINVAL               # boatagent_collect's own checks still apply
    torch.cuda.synchronize()
    assert mem.mem_cntr == 0
    assert same(state_part(env), before[0]) and same(env.obs, before[1]) and torch.equal(rec._buf, before[2])
    assert call(steps=8) == 0                    # exactly the capacity: accepted
    torch.cuda.synchronize()
    assert mem.mem_cntr == 8 * 64
    for x in (env, env64, fresh, mem):
        x.close()


@pytest.mark.gpu
def test_collect_record_value_errors(S, tmp_path):
    import torch
    pol = policy(make_actor(seed=1))
    env, other = make_env(S, 6, 64), make_env(S, 6, 64)
    mem = make_ring(S, 10_000)
    rec = S.DeviceRecorder(env, [1, 2], str(tmp_path / "a"), capacity=8)
    rec_other = S.DeviceRecorder(other, [1, 2], str(tmp_path / "b"), capacity=8)
    rec.start()
    pol.collect(env, mem, 4, recorder=rec)
    torch.cuda.synchronize()
    before = rec.pending, pol.steps, mem.mem_cntr, state_part(env).clone()
    with pytest.raises(ValueError):
        pol.collect(env, mem, 4, recorder=rec_other)
    with pytest.raises(ValueError):
        pol.collect(env, mem, 9, recorder=rec)
    assert (rec.pending, pol.steps, mem.mem_cntr) == before[:3] and same(state_part(env), before[3])
    rec.close()
    rec_other.close()
    for x in (env, other, mem):
        x.close()


# ---------------------------------------------------------------------------------------
# 8. CPU: the recording instantiations compile without spills and fit the launch bound
# ---------------------------------------------------------------------------------------
def test_recording_collect_kernels_compile_without_spills(tmp_path):
    from sac_agent_b200 import _build
    src = os.path.join(_build.CSRC, "rollout.cu")
    r = subprocess.run([_build.nvcc(), "-Xptxas=-v", *_build.ARCH, *_build.COMMON, "-c", src, "-o",
                        str(tmp_path / "rollout.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    blocks = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads\n[^\n]*Used (\d+) registers", r.stderr)
    record = {re.search(r"collect_kernelILi(\d)ELb1E", b[0]).group(1): b[1:] for b in blocks
              if re.search(r"collect_kernelILi\dELb1E", b[0])}
    assert sorted(record) == ["0", "1", "2", "3", "4"], r.stderr
    for wk, (stack, st, ld, regs) in sorted(record.items()):
        print(f"boat_collect_kernel<{wk}, true>: {regs} registers, {stack} bytes stack, {st}/{ld} spill bytes")
        assert (stack, st, ld) == ("0", "0", "0"), (wk, stack, st, ld)
        assert int(regs) * 288 <= 65536, (wk, regs)   # kThreads = 288 threads, one CTA per SM
