"""The device random streams against the host Philox reference of boat_testlib: the acting draws of the tcgen05 policy
and collect kernels, the replay sample indices (solo and population gathers) and the uniform(-1, 1) action fill.
DESIGN.md ("Random streams") lists each stream's counter, key and conversion; boat_testlib.acting_normal,
replay_indices and uniform_actions state them the way the kernels form the numbers, and these tests hold the kernels to
them value for value: the indices and the fill exactly, the Box-Muller draws to a few fp32 ulps (logf, cospif, expf
and tanhf are the device's few-ulp functions; the build has no fast-math).

The rollout kernel draws through the same actor_normal_draw as the policy kernel and is tied to it bit for bit by
test_gpu_rollout.py::test_rollout_matches_per_step_path, so it needs no case here.

CPU tests: the reference against the Random123 known answers, and the hard-coded edge draws against their edges.
Everything else needs a B200 and is ``@pytest.mark.gpu``."""
import numpy as np
import pytest

from boat_testlib import (acting_normal, acting_words, cospi, philox4x32_10, replay_indices, set_mem_cntr,
                          uniform_actions)

# Actions of the zero-head actor against the float64 reference: 8 fp32 ulps relative (2^-23 |ref| each), the sum of
# the documented bounds of logf, sqrtf, cospif, expf, tanhf and the four roundings in between.
RTOL = 8 * 2.0 ** -23

# (seed, handle row, step, action) of acting draws at the edges of the uniform conversion, found with acting_words.
EDGES = {
    "u1_one": (0x5AC, 0, 3_896_490, 0),      # x >> 8 == 0xFFFFFF: 16777215 + 0.5 rounds to 2^24 in fp32, u1 = 1, e = -0
    "u1_least": (0x5AC, 30, 713_534, 0),     # x >> 8 == 0: u1 = 2^-25, radius sqrt(50 ln 2) = 5.89, e = -5.67
    "cos_zero": (0x5AC, 0, 22_081_522, 0),   # y >> 8 == 2^22 - 1: u2 = 1/4 - 2^-25, cos(2 pi u2) = 1.9e-7
    # y >> 8 == 0xC00000: 12582912 + 0.5 rounds to 12582912 in fp32, u2 = 3/4 and cospif(3/2) = 0 exactly, e = 0
    "cos_exact_zero": (0x5AC, 44_588, 2 ** 32, 3),
}


@pytest.fixture(scope="module")
def S():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import sac_agent_b200 as pkg
    pkg.lib()
    return pkg


# ---------------------------------------------------------------------------------------
# CPU: the reference itself
# ---------------------------------------------------------------------------------------
def test_reference_philox_known_answers_vectorised():
    """The Random123 kat_vectors of philox4x32-10, all three in one broadcast call per key (the key is a scalar), and
    counters wider than 32 bits cut to their low word as the kernels' (uint32_t) casts do."""
    f = 0xFFFFFFFF
    ctr = np.array([[0, 0, 0, 0], [f, f, f, f], [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344]], dtype=np.uint64)
    keys = [(0, 0), (f, f), (0xA4093822, 0x299F31D0)]
    want = [(0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)]
    for k, (key, w) in enumerate(zip(keys, want)):
        out = philox4x32_10(*ctr.T, *key)
        assert tuple(int(x[k]) for x in out) == w
        assert tuple(int(x) for x in philox4x32_10(*(ctr[k] + np.uint64(1 << 32) * np.uint64(7)), *key)) == w


def test_edge_draws_select_their_edges():
    x, y = (int(w) for w in acting_words(*EDGES["u1_one"]))
    assert x >> 8 == 0xFFFFFF and np.float32(x >> 8) + np.float32(0.5) == np.float32(2.0 ** 24)
    assert acting_normal(*EDGES["u1_one"]) == 0.0
    x, y = (int(w) for w in acting_words(*EDGES["u1_least"]))
    assert x >> 8 == 0 and acting_normal(*EDGES["u1_least"]) == pytest.approx(-5.6706, abs=1e-4)
    x, y = (int(w) for w in acting_words(*EDGES["cos_zero"]))
    assert y >> 8 == (1 << 22) - 1 and 0 < acting_normal(*EDGES["cos_zero"]) < 3e-7
    x, y = (int(w) for w in acting_words(*EDGES["cos_exact_zero"]))
    assert y >> 8 == 0xC00000 and np.float32(y >> 8) + np.float32(0.5) == np.float32(0.75 * 2 ** 24)
    assert acting_normal(*EDGES["cos_exact_zero"]) == 0.0


def test_reference_cospi_is_exact_at_the_quarter_turns():
    x = np.array([0.0, 0.5, 1.0, 1.5, 2.0])
    assert np.array_equal(cospi(x), [1.0, 0.0, -1.0, 0.0, 1.0])
    y = np.linspace(0.0, 2.0, 10_001)
    assert np.abs(cospi(y) - np.cos(np.pi * y)).max() < 1e-15


# ---------------------------------------------------------------------------------------
# GPU: acting noise
# ---------------------------------------------------------------------------------------
def zero_head_policy(n_actions, max_action, seed):
    """An actor whose head weights are zero, mean bias 0 and std bias -30: tanhf(-30) = -1, so log_std is exactly -5
    and action = tanh(e exp(-5)) * max_action, nearly linear in the draw e and independent of the bf16 hidden layers."""
    import torch
    from sac_agent_b200.networks import ActorNetwork, TensorCorePolicy
    actor = ActorNetwork(None, (11,), max_action, n_actions=n_actions).cuda()
    with torch.no_grad():
        actor.mean.weight.zero_()
        actor.std.weight.zero_()
        actor.mean.bias.zero_()
        actor.std.bias.fill_(-30.0)
    return TensorCorePolicy(actor, seed=seed)


def squash(e, max_action):
    return np.tanh(e * np.exp(-5.0)) * np.asarray(max_action, dtype=np.float64)


def check_actions(got, ref, what):
    """|got - ref| <= RTOL |ref| everywhere (a zero reference needs a zero action, a NaN or infinite action fails);
    returns the worst error in fp32 ulps (2^-23 relative)."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == np.shape(ref), (what, got.shape, np.shape(ref))
    err = np.abs(got - ref)
    bad = ~(err <= RTOL * np.abs(ref))   # written so that a NaN compares as bad
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        pytest.fail(f"{what}: {int(bad.sum())} of {bad.size} actions off the reference, first at {i}: "
                    f"got {got[i]!r}, reference {ref[i]!r}")
    nz = ref != 0
    return float((err[nz] / np.abs(ref[nz])).max() / 2.0 ** -23) if nz.any() else 0.0


def test_check_actions_rejects_nan_inf_and_off_values():
    """The comparison behind the acting-noise tests: the float32 rounding of the reference passes; a NaN (what logf of
    a u1 above 1 would give), an infinity, a value 16 ulps off or a non-zero action for a zero draw each fail."""
    ref = squash(acting_normal(0x5AC, np.arange(1000)[None, :], np.arange(3)[:, None], 0), 1.0)
    ref[1, 7] = 0.0
    assert check_actions(ref.astype(np.float32), ref, "fp32 rounding") <= 1.0
    nan_everywhere = np.full_like(ref, np.nan)
    for i, v in (((0, 0), np.nan), ((2, 999), np.inf), ((1, 3), ref[1, 3] * (1 + 16 * 2.0 ** -23)), ((1, 7), 1e-30)):
        got = ref.copy()
        got[i] = v
        with pytest.raises(pytest.fail.Exception):
            check_actions(got, ref, "one bad action")
    with pytest.raises(pytest.fail.Exception):
        check_actions(nan_everywhere, ref, "all NaN")


MAX_ACTIONS = [1.0, 0.5, 2.0, 0.75, 1.5, 0.25, 3.0, 0.125]


@pytest.mark.gpu
@pytest.mark.parametrize("n_actions", [1, 2, 4, 8])
def test_policy_act_draws_match_reference(S, n_actions):
    """boatagent_policy_act without eps: action (row, a) at call `steps` is the draw of (seed; row, steps, a).  Ragged
    tiles and several tiles per CTA, step counters across the 2^32 boundary, seeds with a high key word."""
    import torch
    ns, big = (1, 127, 128, 129), 70_001
    max_a = np.array(MAX_ACTIONS[:n_actions], dtype=np.float32)
    obs = torch.rand(big, 11, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n_actions))
    rows, acts = np.arange(big)[:, None], np.arange(n_actions)[None, :]
    worst = 0.0
    for seed in (0, 0x5AC, 2 ** 40 + 9):
        pol = zero_head_policy(n_actions, max_a, seed)
        for step in (0, 5, 2 ** 32 - 1, 2 ** 32, 2 ** 40 + 3):
            ref = squash(acting_normal(seed, rows, step, acts), max_a)
            for n in ns + (big,):
                pol.steps = step
                got = pol.act(obs[:n]).cpu().numpy()
                assert pol.steps == step + 1
                worst = max(worst, check_actions(got, ref[:n], f"seed {seed:#x}, step {step}, n {n}"))
    print(f"policy_act n_actions={n_actions}: worst action error {worst:.2f} fp32 ulps")


@pytest.mark.gpu
def test_policy_act_edge_draws(S):
    """The draws at the ends of the uniform conversion: u1 = 1 (the draw is -0, so is the action), the least u1 (the
    largest radius), u2 next to 1/4 (cos next to 0) and u2 = 3/4 (cos exactly 0, so is the action)."""
    import torch
    for name, (seed, row, step, a) in EDGES.items():
        n_actions = next(k for k in (1, 2, 4, 8) if k > a)
        pol = zero_head_policy(n_actions, [1.0] * n_actions, seed)
        pol.steps = step
        got = pol.act(torch.rand(row + 1, 11, device="cuda")).cpu().numpy()[row, a]
        check_actions(np.array([got]), np.array([squash(acting_normal(seed, row, step, a), 1.0)]), name)


@pytest.mark.gpu
def test_policy_act_matches_injected_reference_draws(S):
    """A trained-looking actor (default init: live mean and std heads): act(obs) is act(obs, eps) with eps the float32
    reference draws of the same (seed, row, step, action)."""
    import torch
    from sac_agent_b200.networks import ActorNetwork, TensorCorePolicy
    torch.manual_seed(5)
    seed, n = 2 ** 40 + 9, 1000
    actor = ActorNetwork(None, (11,), [1.0, 0.5], n_actions=2).cuda()
    pol = TensorCorePolicy(actor, seed=seed)
    obs = torch.rand(n, 11, device="cuda")
    for step in (7, 2 ** 32 + 1):
        pol.steps = step
        drawn = pol.act(obs).clone()
        eps = acting_normal(seed, np.arange(n)[:, None], step, np.arange(2)[None, :]).astype(np.float32)
        pol.steps = step
        injected = pol.act(obs, torch.from_numpy(eps).cuda())
        assert float((drawn - injected).abs().max()) <= 1e-6, step


@pytest.mark.gpu
@pytest.mark.parametrize("n_envs,env_id_offset", [(1000, 0), (70_001, 0), (1000, 1000)])
def test_collect_draws_match_reference(S, n_envs, env_id_offset):
    """boatagent_collect: the action of ring row (step t, env i) is the draw of (seed; i, step0 + t), i the row of the
    handle whatever its env_id_offset; the call crosses the 2^32 boundary of the step counter."""
    import torch
    seed, T, step0 = 0x5AC, 3, 2 ** 32 - 2
    pol = zero_head_policy(1, [1.0], seed)
    env = S.BatchedBoatEnv(S.load_config(base_settings__experiment=6), n_envs, seed=3, precision="fp32", device=0,
                           env_id_offset=env_id_offset, auto_reset=True)
    env.reset()
    mem = S.ReplayBuffer(T * n_envs, (11,), 1, precision="fp32", device=0, as_torch=True)
    pol.steps = step0
    pol.collect(env, mem, T)
    assert pol.steps == step0 + T and mem.mem_cntr == T * n_envs
    got = mem.gather(torch.arange(T * n_envs, device="cuda"))[1].cpu().numpy().reshape(T, n_envs)
    ref = squash(acting_normal(seed, np.arange(n_envs)[None, :], step0 + np.arange(T)[:, None], 0), 1.0)
    worst = check_actions(got, ref, f"collect n {n_envs}, offset {env_id_offset}")
    print(f"collect n={n_envs} offset={env_id_offset}: worst action error {worst:.2f} fp32 ulps")
    env.close()
    mem.close()


# ---------------------------------------------------------------------------------------
# GPU: replay sample indices
# ---------------------------------------------------------------------------------------
RING = 12_000_000
BATCHES = (1, 3, 4, 5, 127, 128, 129, 4096, 700_003)   # 700,003 > 4736 CTAs x 128 rows: the grid-stride loop runs


@pytest.fixture(scope="module")
def big_ring(S):
    ring = S.ReplayBuffer(RING, (1,), 1, precision="fp32", device=0, as_torch=True)
    yield ring
    ring.close()


@pytest.mark.gpu
@pytest.mark.parametrize("max_mem,mem_cntr", [(1, 1), (2, 2), (3, 3), (7, 7), (300, 300), (RING, 2 * RING + 12_345),
                                              (10_000_019, 10_000_019)],
                         ids=["1", "2", "3", "7", "300", "wrapped", "partial"])
def test_sample_indices_match_reference(big_ring, max_mem, mem_cntr):
    """sample_buffer(batch, return_indices=True) draws exactly replay_indices(seed, sample counter, batch, max_mem)."""
    set_mem_cntr(big_ring, mem_cntr)
    for seed in (0, 2 ** 40 + 3):
        big_ring.seed = seed
        for counter in (0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 40 + 7):
            ref = replay_indices(seed, counter, BATCHES[-1], max_mem)
            for batch in BATCHES:
                big_ring._samples = counter
                idx = big_ring.sample_buffer(batch, return_indices=True)[-1].cpu().numpy()
                assert big_ring._samples == counter + 1
                assert np.array_equal(idx, ref[:batch]), (seed, counter, batch)


@pytest.mark.gpu
def test_sample_indices_fp64_ring(S):
    ring = S.ReplayBuffer(5000, (11,), 2, precision="fp64", device=0, as_torch=True)
    set_mem_cntr(ring, 4321)
    ring.seed, ring._samples = 2 ** 40 + 3, 2 ** 32
    idx = ring.sample_buffer(4099, return_indices=True)[-1].cpu().numpy()
    assert np.array_equal(idx, replay_indices(2 ** 40 + 3, 2 ** 32, 4099, 4321))
    ring.close()


@pytest.mark.gpu
def test_sample_members_indices_match_reference(S):
    """boatreplay_sample_members has no index output: every row's state is its slot number, so the gathered rows give
    the indices back.  Three rings with their own seeds, counters and fill levels, one of them wrapped."""
    import torch
    from sac_agent_b200 import _lib
    specs = [  # (ring size, rows stored, mem_cntr afterwards, seed, sample counter)
        (1000, 1000, 3 * 1000 + 17, 0, 2 ** 32 - 1),
        (5000, 300, 300, 2 ** 40 + 3, 0),
        (200_003, 150_001, 150_001, 0x5AC, 2 ** 40 + 7),
    ]
    rings = []
    for size, n, cntr, seed, counter in specs:
        r = S.ReplayBuffer(size, (1,), 1, precision="fp32", device=0, as_torch=True)
        s = torch.arange(n, dtype=torch.float32, device="cuda").reshape(n, 1)
        r.store_batch(s, -s, 2 * s.reshape(n), s + 0.5, s.reshape(n) % 3 == 0)
        set_mem_cntr(r, cntr)
        rings.append(r)
    for batch in (129, 700_003):
        outs = [r._outputs(batch) for r in rings]
        tbl = (_lib.SampleMember * len(rings))(*[_lib.SampleMember(r._h, spec[3], spec[4], *[t.data_ptr() for t in o])
                                                 for r, o, spec in zip(rings, outs, specs)])
        assert S.lib().boatreplay_sample_members(tbl, len(rings), batch, None) == 0
        torch.cuda.synchronize()
        for (size, n, cntr, seed, counter), (st, ac, rw, st2, dn) in zip(specs, outs):
            j = st[:, 0]
            assert torch.equal(ac[:, 0], -j) and torch.equal(rw, 2 * j) and torch.equal(st2[:, 0], j + 0.5)
            assert torch.equal(dn.bool(), j % 3 == 0)
            ref = replay_indices(seed, counter, batch, min(cntr, size))
            assert np.array_equal(j.cpu().numpy().astype(np.int64), ref), (size, batch)
    for r in rings:
        r.close()


# ---------------------------------------------------------------------------------------
# GPU: the uniform(-1, 1) action fill
# ---------------------------------------------------------------------------------------
SCALES = (1.0, 0.05, 4.0, 1.0 / 3.0)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_uniform_actions_match_reference(S, precision):
    """env.uniform_actions(step, scale) is uniform_actions(seed, global ids, step, scale) bit for bit: whole handles of
    1 .. 1,000,003 envs, the three shards of 1,000,003 envs (offsets that are not multiples of 4, so a shard's first
    quad straddles its edge) and an out= view one element into a larger tensor (the unaligned scalar path).  The scale
    is rounded to fp32 before the multiply, also for fp64 handles, whose actions are the fp32 values widened."""
    import torch
    dtype = np.float32 if precision == "fp32" else np.float64
    bits = np.int32 if precision == "fp32" else np.int64
    total = 1_000_003
    handles = [(0, n) for n in (1, 3, 5, 1000, total)] + [S.shard_range(total, r, 3) for r in range(3)]
    assert any(off % 4 for off, _ in handles)
    cfg = S.load_config(base_settings__experiment=6)
    for seed in (0, 2 ** 40 + 9):
        refs = {step: uniform_actions(seed, np.arange(total), step, np.array(SCALES)[:, None], np.float32).astype(dtype)
                for step in (0, 7, 2 ** 32 - 1, 2 ** 32, 2 ** 40 + 5)}
        for off, n in handles:
            env = S.BatchedBoatEnv(cfg, n, seed=seed, precision=precision, device=0, env_id_offset=off)
            buf = torch.full((n + 2,), 7.0, dtype=env.dtype, device="cuda")
            for step, ref in refs.items():
                for k, scale in enumerate(SCALES):
                    got = env.uniform_actions(step, scale).cpu().numpy()
                    assert np.array_equal(got.view(bits), ref[k, off:off + n].view(bits)), (seed, off, n, step, scale)
                env.uniform_actions(step, SCALES[-1], out=buf[1:n + 1])
                got = buf.cpu().numpy()
                assert got[0] == 7.0 and got[-1] == 7.0
                assert np.array_equal(got[1:n + 1].view(bits), ref[-1, off:off + n].view(bits)), (seed, off, n, step)
            env.close()
