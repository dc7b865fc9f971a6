"""CPU-only checks of the boundary: libboatenv.so loads without a GPU and exports every
symbol include/boatenv.h declares; the ctypes binding covers exactly that set; host-side
logic (config parsing, Philox draws, error codes, sharding, the gloo all-reduce)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from boat_testlib import philox4x32_10

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "boatenv.h")


@pytest.fixture(scope="module")
def S():
    import sac_agent_b200 as pkg
    from sac_agent_b200 import _build
    _build.build()  # nvcc cross-compiles sm_100a without a GPU; a no-op when up to date
    return pkg


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"BOATENV_API\s+[\w\s\*]+?\b(boat\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol(S):
    names = declared_symbols()
    assert len(names) >= 30
    lib = C.CDLL(S.library_path())
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/boatenv.h but not exported"
    from sac_agent_b200 import _lib
    assert sorted(_lib.SIGNATURES) == names  # the binding covers the header, no more, no less
    # nothing but the C ABI is exported (hidden visibility for the C++ internals)
    out = subprocess.run(["nm", "-D", "--defined-only", S.library_path()], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert exported == set(names), exported ^ set(names)


def test_version_and_error_strings(S):
    L = S.lib()
    assert b"sm_100a" in L.boatenv_version()
    assert L.boatenv_error_string(0) == b"ok"
    assert b"experiment" in L.boatenv_error_string(-2)
    assert b"fixed_points" in L.boatenv_error_string(-3)
    assert L.boatenv_kernel_launches() >= 0


def test_no_cpu_fallback_without_device(S):
    """Without a CUDA device the product path refuses to run (no CPU fallback)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError):
        S.BatchedBoatEnv(S.load_config(), 4)
    with pytest.raises(RuntimeError):
        S.ReplayBuffer(16, (11,), 1)
    # and the C ABI itself answers BOATENV_ENODEVICE
    h = C.c_void_p()
    p = S.params_from_config(S.load_config())
    assert S.lib().boatenv_create(C.byref(p), 4, 0, 0, 32, 0, C.byref(h)) == -5
    assert S.lib().boatreplay_create(16, 11, 1, 32, 0, C.byref(h)) == -5
    arr = (C.c_double * 4)(10, 10, 0.01, 0.1)
    assert S.lib().boattoy_create(0, 4, arr, 4, 0.0, 0, 32, 0, C.byref(h)) == -5


def test_missing_library_fails_loudly(S, monkeypatch):
    from sac_agent_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "_LIB_NAME", "libboatenv_missing.so")
    with pytest.raises(ImportError, match="no CPU fallback"):
        _lib.lib()


def test_config_semantics(S, tmp_path):
    """A reference YAML (original_config.yaml) is accepted unchanged; only the hot-path keys are read;
    the built-in defaults equal the reference's shipped values (as recorded in tests/golden)."""
    import yaml
    from boat_testlib import reference_config_record
    cfg = S.load_config()
    p = S.params_from_config(cfg)
    assert (p.dt, p.t_max, p.track_width, p.goal_line, p.fuel) == (0.25, 2500.0, 800.0, 3900.0, 15000.0)
    assert (p.fixed_points, p.max_velocity, p.direction) == (8, 0.5, 90.0)
    theirs = reference_config_record()
    theirs["base_settings"]["experiment"] = cfg.base_settings.experiment   # not recorded: every roll-out sets its own
    q = S.params_from_config(theirs)
    for name, _ in p._fields_:
        assert getattr(p, name) == getattr(q, name), name
    ref_cfg = tmp_path / "original_config.yaml"
    ref_cfg.write_text(yaml.safe_dump(theirs))
    r = S.params_from_config(S.load_config(str(ref_cfg)))  # the reference's values as a YAML file, read by our loader
    assert bytes(memoryview(r).cast("B")) == bytes(memoryview(q).cast("B"))
    # plain dicts and attribute containers both work (the reference passes a DotMap)
    assert S.params_from_config(dict(cfg)).boat_m == p.boat_m
    assert cfg.base_settings.experiment == cfg["base_settings"]["experiment"]
    assert S.load_config(base_settings__experiment=5).base_settings.experiment == 5


def philox_words(*ctr_and_key):
    return tuple(int(w) for w in philox4x32_10(*ctr_and_key))


def test_philox_known_answers():
    """Random123 kat_vectors for philox4x32-10."""
    assert philox_words(0, 0, 0, 0, 0, 0) == (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)
    f = 0xffffffff
    assert philox_words(f, f, f, f, f, f) == (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)
    assert philox_words(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0xa4093822, 0x299f31d0) == \
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)


def test_host_philox_draws(S):
    """boatenv_episode_draws_host: np.random.randint(-640, 640) / np.random.sample(8)
    stand-ins, a pure function of (seed, global env id, episode)."""
    L = S.lib()
    p = S.params_from_config(S.load_config(base_settings__experiment=6))

    def draws(seed, env, ep):
        s = C.c_int32()
        k = (C.c_double * 16)()
        assert L.boatenv_episode_draws_host(C.byref(p), seed, env, ep, C.byref(s), k) == 0
        return s.value, np.array(k[:])

    a = draws(1, 12345, 3)
    assert a[0] == draws(1, 12345, 3)[0] and np.array_equal(a[1], draws(1, 12345, 3)[1])
    assert not np.array_equal(a[1], draws(1, 12345, 4)[1]) and not np.array_equal(a[1], draws(2, 12345, 3)[1])
    assert not np.array_equal(a[1], draws(1, 12346, 3)[1])
    sy = np.array([draws(7, e, 0)[0] for e in range(4000)])
    assert sy.min() >= -640 and sy.max() < 640 and abs(sy.mean()) < 30 and sy.std() == pytest.approx(369.5, rel=0.05)
    kn = np.concatenate([draws(7, e, 0)[1] for e in range(500)])
    assert kn.min() > 0 and kn.max() < 1 and abs(kn.mean() - 0.5) < 0.02
    assert np.array_equal(kn, kn.astype(np.float32).astype(np.float64))  # exact in fp32
    # independent Philox4x32-10 (pinned by the Random123 known answers below) + the documented
    # counter layout (env_lo, env_hi, episode, block) / key (seed_lo, seed_hi) reproduce the draws
    for seed, env, ep in ((1, 12345, 3), (2 ** 40 + 5, 2 ** 33 + 7, 9)):
        s_y, knots = draws(seed, env, ep)
        key = (seed & 0xffffffff, seed >> 32)
        w0 = philox_words(env & 0xffffffff, env >> 32, ep, 0, *key)[0]
        assert s_y == -640 + ((w0 * 1280) >> 32)
        for t in range(16):
            w = philox_words(env & 0xffffffff, env >> 32, ep, 1 + (t >> 2), *key)[t & 3]
            assert knots[t] == ((((w >> 9) << 1) | 1) / 16777216.0)
    bad = S.params_from_config(S.load_config(base_settings__experiment=9))
    assert L.boatenv_episode_draws_host(C.byref(bad), 0, 0, 0, None, None) == -2
    few = S.params_from_config(S.load_config(base_settings__experiment=4, wind__fixed_points=3))
    assert L.boatenv_episode_draws_host(C.byref(few), 0, 0, 0, None, None) == -3


def test_shard_range_tiles_population(S):
    for n_total in (0, 1, 7, 4096, 16_777_216, 1_000_003):
        for world in (1, 2, 3, 4, 8):
            spans = [S.shard_range(n_total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and sum(c for _, c in spans) == n_total
            for (o1, c1), (o2, _) in zip(spans, spans[1:]):
                assert o1 + c1 == o2
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1
    with pytest.raises(ValueError):
        S.shard_range(10, 2, 2)


def test_host_batch_draws_equal_the_per_pair_draws(S):
    """boatenv_episode_draws_batch_host == boatenv_episode_draws_host for every (env, episode) of the batch."""
    L = S.lib()
    p = S.params_from_config(S.load_config(base_settings__experiment=6))
    ids = np.array([0, 1, 31, 32, 12345, 2 ** 33 + 7], dtype=np.int64)
    E, e0 = 5, 3
    s_y = np.empty((E, len(ids)), dtype=np.int32)
    knots = np.empty((E, len(ids), 2, 8))
    assert L.boatenv_episode_draws_batch_host(C.byref(p), 9, ids.ctypes.data, len(ids), e0, E, s_y.ctypes.data,
                                              knots.ctypes.data) == 0
    for e in range(E):
        for j, g in enumerate(ids):
            s = C.c_int32()
            k = (C.c_double * 16)()
            assert L.boatenv_episode_draws_host(C.byref(p), 9, int(g), e0 + e, C.byref(s), k) == 0
            assert s.value == s_y[e, j] and np.array_equal(np.array(k[:]).reshape(2, 8), knots[e, j])
    assert L.boatenv_episode_draws_batch_host(C.byref(p), 9, None, 1, 0, 1, None, None) == -1
    neg = np.array([-1], dtype=np.int64)
    assert L.boatenv_episode_draws_batch_host(C.byref(p), 9, neg.ctypes.data, 1, 0, 1, s_y.ctypes.data, None) == -1


def test_host_toy_parameters(S):
    """boattoy_params_host: env 0 keeps the script constants (toy_car.py:7-8,11,23; toy_parachute.py:8-15), every
    other env gets each constant times (1 + jitter * u), u in [-1, 1) from Philox(seed, env, parameter)."""
    L = S.lib()
    car = np.array([10.0, 10.0, 0.01, 0.1])
    out = np.empty((1000, 4))
    arr = (C.c_double * 4)(*car)
    assert L.boattoy_params_host(0, arr, 4, 0.1, 3, 0, 1000, out.ctypes.data) == 0
    assert np.array_equal(out[0], car) and np.all(np.abs(out[1:] / car - 1.0) <= 0.1)
    assert np.unique(out[:, 0]).size > 990 and abs((out[1:, 0] / 10.0 - 1.0).mean()) < 0.01
    again = np.empty((10, 4))
    assert L.boattoy_params_host(0, arr, 4, 0.1, 3, 500, 10, again.ctypes.data) == 0
    assert np.array_equal(again, out[500:510])                       # a pure function of (seed, env, parameter)
    other = np.empty((10, 4))
    assert L.boattoy_params_host(0, arr, 4, 0.1, 4, 500, 10, other.ctypes.data) == 0 and not np.array_equal(other, again)
    flat = np.empty((5, 4))
    assert L.boattoy_params_host(0, arr, 4, 0.0, 3, 0, 5, flat.ctypes.data) == 0 and np.all(flat == car)
    assert L.boattoy_params_host(0, arr, 9, 0.1, 3, 0, 5, flat.ctypes.data) == -1     # wrong parameter count for a car
    assert L.boattoy_params_host(7, arr, 4, 0.1, 3, 0, 5, flat.ctypes.data) == -1     # unknown toy


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
import sac_agent_b200 as S
from sac_agent_b200.sharding import dist_info
rank, local_rank, world = dist_info()
dist.init_process_group("gloo", rank=rank, world_size=world)
off, n = S.shard_range(1000, rank, world)
# each rank's statistics vector: what BatchedBoatEnv.counters_tensor() yields on a GPU rank
c = torch.tensor([rank + 1, 2, 0, 0, 10 * (rank + 1), 12 + 11 * rank, -5.0 * (rank + 1), 40.0], dtype=torch.float64)
out = S.all_reduce_counters(c)
spans = [None] * world
dist.all_gather_object(spans, (off, n))
if rank == 0:
    assert spans == [(0, 500), (500, 500)], spans
    assert out["reached_goal"] == 3 and out["rudder_broken"] == 30 and out["episodes"] == 35, out
    assert out["return_sum"] == -15.0 and abs(out["return_mean"] + 15.0 / 35) < 1e-12, out
    print("GLOO_OK")
dist.destroy_process_group()
"""


def test_world_size_2_gloo_all_reduce(S, tmp_path):
    """The N>1 path on CPU: two processes, gloo, contiguous shards + the statistics all-reduce."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "GLOO_OK" in r.stdout


_PBT_WORKER = """
import random, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
from sac_agent_b200 import population as P
from sac_agent_b200.sharding import dist_info
rank, local_rank, world = dist_info()
dist.init_process_group("gloo", rank=rank, world_size=world)
# member r: weights filled with r, an int64 step counter, its own hyper-parameters; rank 1 has the better score
tensors = [torch.full((3, 4), float(rank)), torch.full((5,), 10.0 * rank), torch.tensor([100 + rank, 7], dtype=torch.int64)]
hp = dict(alpha=0.002 + 0.004 * rank, beta=0.001 + 0.002 * rank, gamma=0.97, tau=0.005)
new_hp, info = P.exploit_explore(tensors, hp, score=[-500.0, -100.0][rank], rng=random.Random(5), bottom_fraction=0.25)
assert info["ranking"] == [1, 0] and info["scores"] == [-500.0, -100.0], info
if rank == 0:   # the loser adopted member 1's state and a perturbed copy of its hyper-parameters
    assert info["adopted_from"] == 1
    assert torch.equal(tensors[0], torch.ones(3, 4)) and torch.equal(tensors[1], torch.full((5,), 10.0))
    assert tensors[2].tolist() == [101, 7] and tensors[2].dtype == torch.int64
    for k, (lo, hi) in P.HP_RANGES.items():
        assert lo <= new_hp[k] <= hi
    assert new_hp["alpha"] in (round(0.006 * 0.8, 4), round(0.006 * 1.25, 4)), new_hp
    assert new_hp["gamma"] in (round(1 - 0.03 * 0.8, 4), round(1 - 0.03 * 1.25, 4)), new_hp
else:           # the winner is untouched
    assert info["adopted_from"] is None and new_hp == hp and torch.equal(tensors[0], torch.ones(3, 4))
# a round in which nobody finished an episode changes nothing
hp2, info2 = P.exploit_explore(tensors, new_hp, score=float("nan"), rng=random.Random(6))
assert info2["adopted_from"] is None and hp2 == new_hp
dist.barrier()
if rank == 0:
    print("PBT_OK")
dist.destroy_process_group()
"""


def test_population_exploit_explore_world_size_2_gloo(S, tmp_path):
    """SURVEY.md 8f rank 3: the exploit / explore round of population-based training on two gloo ranks."""
    script = tmp_path / "pbt_worker.py"
    script.write_text(_PBT_WORKER.format(root=ROOT))
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "PBT_OK" in r.stdout


def test_population_perturb_stays_in_the_tuner_ranges():
    import random
    sys.path.insert(0, ROOT)
    from sac_agent_b200 import population as P
    rng = random.Random(0)
    hp = dict(alpha=0.01, beta=0.0008, gamma=0.99, tau=0.001)
    for _ in range(50):
        hp = P.perturb(hp, rng)
        for k, (lo, hi) in P.HP_RANGES.items():
            assert lo <= hp[k] <= hi and round(hp[k], 4) == hp[k]
